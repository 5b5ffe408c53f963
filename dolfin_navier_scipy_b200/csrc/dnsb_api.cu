// dnsb_api.cu -- C ABI of libdnsb200.so (see include/dnsb.h)
//
// Build:  nvcc -shared -Xcompiler -fPIC -O3 -lineinfo
//              -gencode arch=compute_100a,code=sm_100a  dnsb_api.cu -o libdnsb200.so
#include "../../include/dnsb.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <new>

#include "dnsb_common.cuh"
#include <cuda.h>
#ifdef DNSB_NO_NC
// experiment: no read-only (ld.global.nc) loads -- see DESIGN.md, programmatic dependent launch
#define __restrict__
#endif
#include "dnsb_kernels.cuh"
#include "dnsb_batched.cuh"
#include "dnsb_dense.cuh"
#include "dnsb_stream.cuh"
#include "dnsb_tc.cuh"
#include "dnsb_tile.cuh"

#define DNSB_VERSION 100

// ===========================================================================
// launch helpers
// ===========================================================================
#define LAUNCH(ctx, kern, grid, block, smem, ...)                              \
  do {                                                                         \
    dnsb_ctx *c_ = (ctx);                                                      \
    const bool pr_ = c_->prof && c_->recs.size() < c_->prof_cap;               \
    cudaEvent_t pe0_ = nullptr, pe1_ = nullptr;                                \
    if (pr_) {                                                                 \
      cudaEventCreate(&pe0_);                                                  \
      cudaEventCreate(&pe1_);                                                  \
      cudaEventRecord(pe0_, c_->stream);                                       \
    }                                                                          \
    {                                                                          \
      cudaLaunchConfig_t cfg_ = {};                                            \
      cfg_.gridDim = dim3(grid);                                               \
      cfg_.blockDim = dim3(block);                                             \
      cfg_.dynamicSmemBytes = (smem);                                          \
      cfg_.stream = c_->stream;                                                \
      cudaLaunchAttribute at_[1];                                              \
      at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;          \
      at_[0].val.programmaticStreamSerializationAllowed = 1;                   \
      cfg_.attrs = at_;                                                        \
      cfg_.numAttrs = (c_->pdl && !pr_ && g_pdl_chain_stream == c_->stream && \
                       (c_->pdl > 1 || (!strstr(#kern, "k_gs_tma") && !strstr(#kern, "k_reduce_partials2"))) && \
                       (c_->pdl_only.empty() || strstr(#kern, c_->pdl_only.c_str())) && \
                       (c_->pdl_skip.empty() || !strstr(#kern, c_->pdl_skip.c_str()))) ? 1 : 0; \
      cudaLaunchKernelEx(&cfg_, kern, __VA_ARGS__);                            \
      g_pdl_chain_stream = pr_ ? nullptr : c_->stream;                         \
    }                                                                          \
    if (pr_) {                                                                 \
      cudaEventRecord(pe1_, c_->stream);                                       \
      c_->recs.push_back(ProfRec{#kern, pe0_, pe1_, c_->next_work});           \
    }                                                                          \
    c_->next_work = 0;                                                         \
    c_->launches++;                                                            \
  } while (0)

// Runtime flags and values to template arguments.  Each instantiation gets a LAUNCH of its own because
// #kern, spelled as written here, is the kernel's name in the profile, which bench.py and the tests match on.
//   LAUNCH_IF(ctx, c, K1, K0, ...)            K1 if c, else K0
//   LAUNCH_B(ctx, K, b, ...)                  K<b>
//   LAUNCH_BB(ctx, K, b0, b1, ...)            (K<b0, b1>)
//   LAUNCH_XBB(ctx, K, X, b0, b1, ...)        (K<X, b0, b1>) for a constant X
//   LAUNCH_BBB(ctx, K, b0, b1, b2, ...)       (K<b0, b1, b2>)
//   LAUNCH_N3(ctx, K, c0, a, c1, b, c, ...)   K<a> if c0, else K<b> if c1, else K<c>; LAUNCH_N4 likewise
#define LAUNCH_IF(ctx, c, K1, K0, ...) \
  do { if (c) LAUNCH(ctx, K1, __VA_ARGS__); else LAUNCH(ctx, K0, __VA_ARGS__); } while (0)
#define LAUNCH_B(ctx, K, b, ...) LAUNCH_IF(ctx, b, K<true>, K<false>, __VA_ARGS__)
#define LAUNCH_BB(ctx, K, b0, b1, ...)                                                   \
  do {                                                                                   \
    if (b0) LAUNCH_IF(ctx, b1, (K<true, true>), (K<true, false>), __VA_ARGS__);         \
    else LAUNCH_IF(ctx, b1, (K<false, true>), (K<false, false>), __VA_ARGS__);          \
  } while (0)
#define LAUNCH_XBB(ctx, K, X, b0, b1, ...)                                               \
  do {                                                                                   \
    if (b0) LAUNCH_IF(ctx, b1, (K<X, true, true>), (K<X, true, false>), __VA_ARGS__);   \
    else LAUNCH_IF(ctx, b1, (K<X, false, true>), (K<X, false, false>), __VA_ARGS__);    \
  } while (0)
#define LAUNCH_BBB(ctx, K, b0, b1, b2, ...)                                              \
  do {                                                                                   \
    if (b0) LAUNCH_XBB(ctx, K, true, b1, b2, __VA_ARGS__);                               \
    else LAUNCH_XBB(ctx, K, false, b1, b2, __VA_ARGS__);                                 \
  } while (0)
#define LAUNCH_N3(ctx, K, c0, a, c1, b, c, ...)                                          \
  do {                                                                                   \
    if (c0) LAUNCH(ctx, K<a>, __VA_ARGS__);                                              \
    else LAUNCH_IF(ctx, c1, K<b>, K<c>, __VA_ARGS__);                                    \
  } while (0)
#define LAUNCH_N4(ctx, K, c0, a, c1, b, c2, c, d, ...)                                   \
  do {                                                                                   \
    if (c0) LAUNCH(ctx, K<a>, __VA_ARGS__);                                              \
    else LAUNCH_N3(ctx, K, c1, b, c2, c, d, __VA_ARGS__);                                \
  } while (0)

static inline int pow2_floor(int x) {
  int p = 1;
  while (2 * p <= x) p *= 2;
  return p;
}

struct RedCfg {   // launch shape of the batched reductions / Gram-Schmidt
  int nblocks, rpb, threads, rows_per_block;
  size_t smem;   // of the single-vector reductions (k_dot1)
};

// Block = rpb x nb threads; a block owns `rows_per_block` contiguous rows, a
// thread at most GS_RPT of them; about 4 blocks per SM when n allows.
static RedCfg red_cfg(dnsb_ctx *ctx, int n, int nb) {
  RedCfg c;
  const int tmax = nb == 1 ? 64 : 256;
  c.rpb = pow2_floor(std::max(1, tmax / nb));
  c.threads = c.rpb * nb;
  int rows = (n + 4 * ctx->sm_count - 1) / (4 * ctx->sm_count);
  rows = ((rows + c.rpb - 1) / c.rpb) * c.rpb;
  rows = std::max(c.rpb, std::min(rows, c.rpb * GS_RPT));
  c.rows_per_block = rows;
  c.nblocks = std::max(1, (n + rows - 1) / rows);
  c.smem = (size_t)c.threads * sizeof(double);
  return c;
}

// TMA-streamed Gram-Schmidt kernels (dnsb_stream.cuh): stages of the basis ring that fit beside the
// reduction scratch in 111 KB (two CTAs per SM); 0 = use the register-pipelined kernels
static int g_gs_tma = 1;
static int gst_stages(const RedCfg &rc, int nb, size_t scratch_doubles) {
  if (!g_gs_tma || nb % 2 || nb < 16 || rc.threads % 32 || rc.threads > 256 ||
      rc.rows_per_block > rc.rpb * GST_RPT)
    return 0;
  const size_t tile = (size_t)rc.rows_per_block * nb * sizeof(double);
  const size_t budget = 111 * 1024, scratch = scratch_doubles * sizeof(double);
  if (scratch + 2 * tile > budget) return 0;
  return (int)std::min<size_t>(GST_MAX_STAGES, (budget - scratch) / tile);
}
static size_t gst_smem(const RedCfg &rc, int nb, int stages, size_t scratch_doubles) {
  return ((size_t)stages * rc.rows_per_block * nb + scratch_doubles) * sizeof(double);
}

// vnext = w - sum_i h[i,m] V_i ; partial2[b*nb + m] = |vnext|^2 over the chunk of block b
static void gs_update_dev(dnsb_ctx *ctx, const RedCfg &rc, const double *V, size_t vstride, int nvec,
                          const double *h, const double *w, double *vnext, int n, int nb,
                          double *partial2, const double *scale = nullptr) {
  const int st = nvec > 0 ? gst_stages(rc, nb, rc.threads) : 0;
  ctx->next_work = nvec;
  if (st >= 2)
    LAUNCH(ctx, k_gs_tma<true>, rc.nblocks, rc.threads + 32, gst_smem(rc, nb, st, rc.threads), V, vstride,
           nvec, h, w, vnext, n, nb, rc.rpb, rc.rows_per_block, partial2, st, scale);
  else
    LAUNCH(ctx, k_gs_update_b, rc.nblocks, rc.threads, rc.smem, V, vstride, nvec, h, w, vnext, n, nb,
           rc.rpb, rc.rows_per_block, partial2, scale);
}

// h[0..nvec) = <V_i, w>, h[nvec] = <w, w>  (per member), deterministic
static void mdot_dev(dnsb_ctx *ctx, const RedCfg &rc, const double *V, size_t vstride,
                     int nvec, const double *w, int n, int nb, double *partial,
                     double *h) {
  const size_t smem = (size_t)(nvec + 1) * rc.threads * sizeof(double);
  const int st = nvec > 0 ? gst_stages(rc, nb, (size_t)(nvec + 1) * rc.threads) : 0;
  ctx->next_work = nvec;
  if (st >= 2)
    LAUNCH(ctx, k_gs_tma<false>, rc.nblocks, rc.threads + 32,
           gst_smem(rc, nb, st, (size_t)(nvec + 1) * rc.threads), V, vstride, nvec, (const double *)nullptr, w,
           (double *)nullptr, n, nb, rc.rpb, rc.rows_per_block, partial, st, (const double *)nullptr);
  else
    LAUNCH(ctx, k_mdot_b, rc.nblocks, rc.threads, smem, V, vstride, nvec, w, n, nb, rc.rpb,
           rc.rows_per_block, partial);
  const int count = (nvec + 1) * nb;
  LAUNCH(ctx, k_reduce_partials2, cdiv(count, 32), 1024, 0, (const double *)partial, rc.nblocks,
         count, h);
}

// ===========================================================================
// CSR handle
// ===========================================================================
struct dnsb_csr {
  dnsb_ctx *ctx = nullptr;
  int nrows = 0, ncols = 0, nnz = 0;
  DBuf<int> indptr, indices;
  DBuf<double> v1, v2;
  bool has2 = false;
  int npair_rows = 0;   // leading rows that pair up (2k, 2k+1) with identical column lists
  SptPlan spt;          // TMA-staged row tiles (dnsb_stream.cuh)
  TilePlan tile;        // fully staged batched Chebyshev step (dnsb_tile.cuh), built by tile_setup
  DBuf<int> t_uptr, t_rptr, t_runs, t_pidx, t_pidxf, t_truns;
  DBuf<int4> t_tdesc, t_pdesc;
  int t_rmax = 0;
  DBuf<double> t_pval;
  DBuf<float> t_pvalf;       // fp32 copy of the packed entries (smoother inside the preconditioner)
  TileDevF tile_view_f() const {
    TileDevF t;
    t.indptr = indptr.p; t.uptr = t_uptr.p; t.rptr = t_rptr.p; t.runs = t_runs.p; t.pidx = t_pidxf.p; t.pval = t_pvalf.p;
    t.tdesc = t_tdesc.p; t.truns = t_truns.p; t.pdesc = t_pdesc.p; t.rmax = t_rmax;
    t.ntiles = tile.ntiles; t.npairs = tile.npairs; t.umax = tile.umax; t.cap = tile.cap; t.stages = tile.stages_f;
    return t;
  }
  TileDev tile_view() const {
    TileDev t;
    t.indptr = indptr.p; t.uptr = t_uptr.p; t.rptr = t_rptr.p; t.runs = t_runs.p; t.pidx = t_pidx.p; t.pval = t_pval.p;
    t.tdesc = t_tdesc.p; t.truns = t_truns.p; t.pdesc = t_pdesc.p; t.rmax = t_rmax;
    t.ntiles = tile.ntiles; t.npairs = tile.npairs; t.umax = tile.umax; t.cap = tile.cap; t.stages = tile.stages;
    return t;
  }
  // host copies (setup only: assembling the block matrix K, diagonal positions)
  std::vector<int> h_indptr, h_indices;
  std::vector<double> h_v1, h_v2;
  CsrDev view() const {
    CsrDev a;
    a.nrows = nrows; a.ncols = ncols; a.nnz = nnz;
    a.indptr = indptr.p; a.indices = indices.p;
    a.v1 = v1.p; a.v2 = has2 ? v2.p : nullptr;
    return a;
  }
  ~dnsb_csr() { cudaStreamSynchronize(ctx->stream); }   // no buffer is freed under a running kernel
};

template <typename T>
static cudaError_t upload_padded(DBuf<T> &b, const T *h, size_t count, size_t pad, cudaStream_t s) {
  cudaError_t e = b.alloc(count + pad);
  if (e != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(b.p + count, 0, pad * sizeof(T), s)) != cudaSuccess) return e;
  if (count && (e = cudaMemcpyAsync(b.p, h, count * sizeof(T), cudaMemcpyHostToDevice, s)) != cudaSuccess)
    return e;
  return cudaStreamSynchronize(s);   // host buffer is borrowed: finish now
}

static int g_tma_stages = 2;
static int g_tma_rows = 64;
// dynamic shared memory the TMA-staged SpMV kernels opt in to (dnsb_ctx_create);
// spt_plan never plans a ring beyond it
static const size_t SPT_SMEM_OPTIN = 216 * 1024;
static size_t spt_stage_bytes(int cap, bool h2) {
  const size_t off_ip = (size_t)cap * (h2 ? 20 : 12);
  return (off_ip + (SPT_ROWS + 4) * 4 + 127) & ~(size_t)127;
}
// row tiles of the TMA-staged SpMM: the largest 4-entry aligned span of a tile fixes the stage size
static SptPlan spt_plan(int nrows, const int32_t *indptr, bool h2) {
  SptPlan p;
  if (nrows == 0 || indptr[nrows] == 0) return p;
  p.rt = g_tma_rows;
  p.ntiles = (nrows + p.rt - 1) / p.rt;
  int span = 0;
  for (int t = 0; t < p.ntiles; ++t) {
    const int r0 = t * p.rt, r1 = std::min(nrows, r0 + p.rt);
    span = std::max(span, ((indptr[r1] + 3) & ~3) - (indptr[r0] & ~3));
  }
  p.cap = (span + 15) & ~15;
  p.stage_bytes = spt_stage_bytes(p.cap, h2);
  // a short ring per CTA and as many CTAs per SM as fit (the CTAs overlap each other's
  // gather and row-sum phases); 228 KB per SM, 1 KB reserved + 1152 B static per CTA
  p.stages = g_tma_stages;
  p.ctas_per_sm = (int)std::min<size_t>(7, (size_t)233472 / (p.stages * p.stage_bytes + 2304));
  if (p.ctas_per_sm < 1 || (size_t)p.stages * p.stage_bytes > SPT_SMEM_OPTIN) {
    p.ctas_per_sm = 1;
    p.stages = (int)std::min<size_t>(SPT_MAX_STAGES, SPT_SMEM_OPTIN / p.stage_bytes);
    if (p.stages < 2) p.stages = 0;   // tile span too long for a ring: k_spmm<8> serves this operator
  }
  p.smem = p.stages * p.stage_bytes;
  return p;
}

static int csr_build(dnsb_ctx *ctx, int nrows, int ncols, const int32_t *indptr,
                     const int32_t *indices, const double *vals1,
                     const double *vals2, std::unique_ptr<dnsb_csr> &out) {
  DNSB_REQUIRE(ctx, nrows >= 0 && ncols >= 0 && indptr, "bad csr args");
  const int nnz = indptr[nrows];
  DNSB_REQUIRE(ctx, nnz >= 0 && (nnz == 0 || (indices && vals1)), "bad csr data");
  for (int i = 0; i < nrows; ++i)
    DNSB_REQUIRE(ctx, indptr[i] <= indptr[i + 1], "indptr not monotone");
  for (int k = 0; k < nnz; ++k)
    DNSB_REQUIRE(ctx, indices[k] >= 0 && indices[k] < ncols, "column index out of range");
  std::unique_ptr<dnsb_csr> m(new (std::nothrow) dnsb_csr());
  DNSB_REQUIRE(ctx, m != nullptr, "out of host memory");
  m->ctx = ctx; m->nrows = nrows; m->ncols = ncols; m->nnz = nnz;
  m->has2 = vals2 != nullptr;
  for (int r = 0; r + 1 < nrows; r += 2) {
    const int a0 = indptr[r], a1 = indptr[r + 1], a2 = indptr[r + 2];
    if (a1 - a0 != a2 - a1 || a1 == a0 || !std::equal(indices + a0, indices + a1, indices + a1)) break;
    m->npair_rows = r + 2;
  }
  m->spt = spt_plan(nrows, indptr, m->has2);
  m->h_indptr.assign(indptr, indptr + nrows + 1);
  m->h_indices.assign(indices, indices + nnz);
  m->h_v1.assign(vals1, vals1 + nnz);
  if (vals2) m->h_v2.assign(vals2, vals2 + nnz);
  // the bulk copies of the staged kernels read whole 16-byte groups: pad the arrays
  DNSB_CK(ctx, upload_padded(m->indptr, indptr, nrows + 1, 8, ctx->stream));
  DNSB_CK(ctx, upload_padded(m->indices, indices, nnz, 4, ctx->stream));
  DNSB_CK(ctx, upload_padded(m->v1, vals1, nnz, 4, ctx->stream));
  if (vals2) DNSB_CK(ctx, upload_padded(m->v2, vals2, nnz, 4, ctx->stream));
  out = std::move(m);
  return 0;
}

static int g_cheb_f32 = 1;  // fp32 work vectors of the Chebyshev smoother inside the preconditioner (tile path)
static int g_proj_t = 1;   // projection space: directions kept raw + a small triangular factor per member
static int g_pkeep = 0;    // raw solutions the projection space is rebuilt from (0: half of its size)
static int g_tail_warps = 8;   // warps of k_spmm_tile that serve the unpaired tail rows (0: separate k_spmm_b2 launch)
static int g_gs_pyth = 1;   // norm of the orthogonalised Arnoldi vector from Pythagoras (batches, columns < 16)
static int g_tile = 1;   // fully TMA-staged batched Chebyshev step (dnsb_tile.cuh)
static int g_init_tile = 1;    // Chebyshev start of the fp32 smoother as a tile kernel (k_cheb_init_tilef)
static int g_tilef_ctas = 2;   // resident CTAs per SM of the fp32 tile kernel (its ring is small enough for two)
static int g_tile_stages = 3, g_tile_stages_f = 3;   // ring depth of the fp64 / fp32 tile kernels (at most what fits)
static const int TILE_SMEM_OPTIN = 220 * 1024;
// tiles of TILE_RP row pairs: unique x rows, tile-local gather offsets, pair-interleaved values.
// Needs the host copies of the matrix (two value arrays, all rows paired).
// `single`: a matrix with one value array (the gradient block JT): the second coefficient of an entry is zero.
static int tile_setup(dnsb_ctx *ctx, dnsb_csr *m, bool single = false) {
  TilePlan &p = m->tile;
  p.ok = false;
  if (!g_tile || m->npair_rows < 2 || m->h_indptr.empty() || ctx->cc < 100) return 0;
  if (single ? m->has2 : (!m->has2 || m->h_v2.empty())) return 0;
  const int np = m->npair_rows / 2;   // leading paired rows (all of F; the velocity rows of K)
  const std::vector<int> &ip = m->h_indptr, &ix = m->h_indices;
  p.npairs = np;
  p.ntiles = (np + TILE_RP - 1) / TILE_RP;
  const size_t npe = (size_t)m->h_indptr[2 * np] / 2;
  std::vector<int> uptr(p.ntiles + 1, 0), rptr(p.ntiles + 1, 0), runs, ucols, pidx(npe + 8, 0);
  std::vector<double> pval((npe + 8) * 4, 0.0);
  std::vector<int> slot(m->ncols, -1);
  p.umax = 0; p.cap = 0;
  for (int t = 0; t < p.ntiles; ++t) {
    const int p0 = t * TILE_RP, p1 = std::min(np, p0 + TILE_RP);
    // unique columns of the tile, ascending; consecutive columns form one run (one bulk copy)
    ucols.clear();
    for (int q = p0; q < p1; ++q)
      for (int k = ip[2 * q]; k < ip[2 * q + 1]; ++k)
        if (slot[ix[k]] < 0) { slot[ix[k]] = 0; ucols.push_back(ix[k]); }
    std::sort(ucols.begin(), ucols.end());
    for (size_t u = 0; u < ucols.size(); ++u) {
      slot[ucols[u]] = (int)u;
      if (u == 0 || ucols[u] != ucols[u - 1] + 1) {
        runs.push_back(ucols[u]); runs.push_back(1); runs.push_back((int)u);
      } else {
        runs[runs.size() - 2] += 1;
      }
    }
    for (int q = p0; q < p1; ++q) {
      const int L = ip[2 * q + 1] - ip[2 * q];
      const size_t e0 = (size_t)ip[2 * q] / 2;
      for (int k = 0; k < L; ++k) {
        const int ka = ip[2 * q] + k, kb = ka + L;
        pidx[e0 + k] = slot[ix[ka]] * TILE_ROWB;
        pval[(e0 + k) * 4 + 0] = m->h_v1[ka]; pval[(e0 + k) * 4 + 1] = single ? 0.0 : m->h_v2[ka];
        pval[(e0 + k) * 4 + 2] = m->h_v1[kb]; pval[(e0 + k) * 4 + 3] = single ? 0.0 : m->h_v2[kb];
      }
    }
    for (size_t u = 0; u < ucols.size(); ++u) slot[ucols[u]] = -1;
    uptr[t + 1] = uptr[t] + (int)ucols.size();
    rptr[t + 1] = (int)(runs.size() / 3);
    p.umax = std::max(p.umax, (int)ucols.size());
    const int pe0 = ip[2 * p0] / 2, pe1 = ip[2 * p1] / 2;
    p.cap = std::max(p.cap, ((pe1 + 3) & ~3) - (pe0 & ~3));
  }
  const size_t off_val = (size_t)p.umax * TILE_ROWB;
  p.stage_bytes = (off_val + (size_t)p.cap * 36 + 127) & ~(size_t)127;
  p.stage_bytes_f = ((size_t)p.umax * (TILE_ROWB / 2) + (size_t)p.cap * 20 + 127) & ~(size_t)127;
  // ring depth: what fits (the kernels are latency bound per tile: more tiles in flight, more bandwidth)
  p.stages = (int)std::min<size_t>(g_tile_stages, (size_t)TILE_SMEM_OPTIN / p.stage_bytes);
  p.stages_f = (int)std::min<size_t>(g_tile_stages_f, (size_t)TILE_SMEM_OPTIN / p.stage_bytes_f);
  if (p.stages < 2 || p.stages_f < 2) return 0;   // neighbourhoods too large for the ring: row-pair kernels
  p.smem = p.stages * p.stage_bytes;
  p.smem_f = p.stages_f * p.stage_bytes_f;
  if (runs.empty()) return 0;
  {
    // per-tile descriptors and a fixed-stride copy of the run lists (addresses known without a lookup),
    // per-pair descriptors (offset into the staged entries, row length)
    int rmax = 0;
    for (int t = 0; t < p.ntiles; ++t) rmax = std::max(rmax, rptr[t + 1] - rptr[t]);
    if (rmax > 32) return 0;   // one run per producer lane
    std::vector<int4> tdesc(p.ntiles), pdesc(np);
    std::vector<int> truns((size_t)p.ntiles * rmax * 3, 0);
    for (int t = 0; t < p.ntiles; ++t) {
      const int p0 = t * TILE_RP, p1 = std::min(np, p0 + TILE_RP);
      const int pe0 = ip[2 * p0] / 2, pe1 = ip[2 * p1] / 2;
      const int a0 = pe0 & ~3, a1 = (pe1 + 3) & ~3;
      tdesc[t] = make_int4(a0, a1 - a0, uptr[t + 1] - uptr[t], rptr[t + 1] - rptr[t]);
      for (int r = rptr[t]; r < rptr[t + 1]; ++r)
        for (int c = 0; c < 3; ++c) truns[((size_t)t * rmax + (r - rptr[t])) * 3 + c] = runs[3 * r + c];
      for (int q = p0; q < p1; ++q) pdesc[q] = make_int4(ip[2 * q] / 2 - a0, ip[2 * q + 1] - ip[2 * q], 0, 0);
    }
    m->t_rmax = rmax;
    DNSB_CK(ctx, m->t_tdesc.upload(tdesc.data(), tdesc.size(), ctx->stream));
    DNSB_CK(ctx, m->t_pdesc.upload(pdesc.data(), pdesc.size(), ctx->stream));
    DNSB_CK(ctx, m->t_truns.upload(truns.data(), truns.size(), ctx->stream));
  }
  DNSB_CK(ctx, m->t_uptr.upload(uptr.data(), uptr.size(), ctx->stream));
  DNSB_CK(ctx, m->t_rptr.upload(rptr.data(), rptr.size(), ctx->stream));
  DNSB_CK(ctx, m->t_runs.upload(runs.data(), runs.size(), ctx->stream));
  DNSB_CK(ctx, m->t_pidx.upload(pidx.data(), pidx.size(), ctx->stream));
  DNSB_CK(ctx, m->t_pval.upload(pval.data(), pval.size(), ctx->stream));
  {
    std::vector<float> pvalf(pval.size());
    std::vector<int> pidxf(pidx.size());
    for (size_t q = 0; q < pval.size(); ++q) pvalf[q] = (float)pval[q];
    for (size_t q = 0; q < pidx.size(); ++q) pidxf[q] = pidx[q] / 2;   // rows of 256 instead of 512 bytes
    DNSB_CK(ctx, m->t_pvalf.upload(pvalf.data(), pvalf.size(), ctx->stream));
    DNSB_CK(ctx, m->t_pidxf.upload(pidxf.data(), pidxf.size(), ctx->stream));
  }
  p.ok = true;
  return 0;
}

// the batched row kernels pre-multiply column indices by nb in int32
static inline bool batched_ok(const dnsb_csr *A, int nb) {
  return nb > 1 && (size_t)std::max(A->ncols, A->nrows) * nb < ((size_t)1 << 31);
}

// groups of SPB_THREADS (row, member) pairs per CTA of the batched row kernels:
// chunks of about `dnsb_rows_per_cta` rows (L1 reuse of the gathered x rows),
// but not fewer than ~2 CTAs per SM
static int g_rows_per_cta = 4;
static int g_dense_ctas_per_sm = 2;
static int g_graphs = 1;
static int g_schur_tf32 = 0;   // 1: dense Schur inverse applied in 3xTF32 (fp32 copy), see dnsb_dense.cuh
static int g_dmma = 1;   // fp64 tensor-core (DMMA) variant of the dense Schur solve
// 1: dense Schur block on the tcgen05 tensor cores (TF32 operands from an fp32 copy of the inverse,
// fp32 accumulation in TMEM; dnsb_tc.cuh).  Preconditioner block only: FGMRES stays fp64.
static int g_schur_l2keep = 0;   // 1: packed inverse read with an L2 evict_last hint (measured: no effect, the streams of a step flush L2 anyway)
static int g_tc_ctas = 1;   // CTAs per SM of k_schur_tc (2: more K splits on all SMs, half the ring depth each)
static int g_schur_tc = 1;
static const int TC_SMEM_OPTIN = 208 * 1024;
static int g_conv_colours = 0;   // 1: coloured scatter instead of the gather formulation of K1a
static inline int spb_gpc(dnsb_ctx *ctx, int nrows, int nb) {
  const long total = (long)nrows * nb;
  long gpc = std::max<long>(1, ((long)g_rows_per_cta * nb) / SPB_THREADS);
  const long groups = (total + SPB_THREADS - 1) / SPB_THREADS;
  while (gpc > 1 && (groups + gpc - 1) / gpc < 2L * ctx->sm_count) gpc /= 2;
  return (int)gpc;
}
// member-pair kernels (double2 elements): nb even
static int g_pair = 1;
static inline bool pair_ok(const dnsb_csr *A, int nb) {
  return g_pair && batched_ok(A, nb) && nb % 2 == 0;
}
static inline unsigned spb2_grid(int nrows, int nb) {
  return cdiv((size_t)nrows * (nb / 2), SPB_THREADS);
}
// row-pair kernels: member pairs AND the leading rows pair up
static int g_rowpair = 1;
static inline int rowpairs_of(const dnsb_csr *A, int nb) {
  return (g_rowpair && pair_ok(A, nb)) ? A->npair_rows / 2 : 0;
}
static inline unsigned spp_grid(int npairs, int nb) {
  return cdiv((size_t)npairs * (nb / 2), SPB_THREADS);
}
#define D2C(p) reinterpret_cast<const double2 *>(p)
#define D2(p) reinterpret_cast<double2 *>(p)
static inline unsigned spb_grid(int nrows, int nb, int gpc) {
  return cdiv((size_t)nrows * nb, (size_t)SPB_THREADS * gpc);
}

// TMA-staged SpMM (dnsb_stream.cuh): operators too large for L2 residency
static int g_tma_min_rows = 65536;
static inline bool spt_ok(const dnsb_csr *A, int nb) {
  return nb == 1 && A->spt.stages >= 2 && A->nrows >= g_tma_min_rows;
}
template <int EPI>
static void spt_launch_epi(dnsb_ctx *ctx, const dnsb_csr *A, const double *coef, const double *x,
                           const SptEpi &ep) {
  const SptPlan &p = A->spt;
  const unsigned grid = (unsigned)std::min(p.ntiles, ctx->sm_count * p.ctas_per_sm);
  LAUNCH_IF(ctx, A->has2 && coef, (k_spmv_tma<true, EPI>), (k_spmv_tma<false, EPI>), grid, SPT_THREADS, p.smem,
            A->view(), coef, x, ep, p.ntiles, p.cap, p.stages, p.rt);
}
static void spt_launch(dnsb_ctx *ctx, const dnsb_csr *A, const double *coef, const double *x,
                       const double *z, double *y, double alpha, double beta) {
  SptEpi ep{z, nullptr, y, nullptr, nullptr, alpha, beta};
  spt_launch_epi<SPT_AXPBY>(ctx, A, coef, x, ep);
}

// y = alpha*A*x + beta*z  on device pointers
static void spmm_dev(dnsb_ctx *ctx, const dnsb_csr *A, const double *coef,
                     const double *x, const double *z, double *y, int nb,
                     double alpha, double beta) {
  if (A->nrows == 0) return;
  if (spt_ok(A, nb)) {
    spt_launch(ctx, A, coef, x, z, y, alpha, beta);
    return;
  }
  if (pair_ok(A, nb)) {
    const bool h2 = A->has2 && coef;
    const int npairs = rowpairs_of(A, nb);
    const int row_begin = 2 * npairs;
    if (h2 && nb == TILE_NB && A->tile.ok && A->tile.npairs == npairs) {
      // TMA-staged tiles for the paired rows (dnsb_tile.cuh), the member-pair kernel for the tail
      // (running the tail -- the long divergence rows of K, 13 us alone -- on a second stream beside
      // the persistent tile kernel was measured: 1.470 instead of 1.451 ms/step, the tile kernel's
      // shared memory leaves no room for a second resident CTA)
      const unsigned grid_ = std::min(A->tile.ntiles, ctx->sm_count);
      const TileDev tv = A->tile_view();
      const int ntw = row_begin < A->nrows ? g_tail_warps : 0;
      const int threads_ = TILE_THREADS + 32 * ntw;
      LAUNCH_B(ctx, k_spmm_tile, beta != 0.0, grid_, threads_, A->tile.smem, tv, coef, x, z, y, alpha, beta,
               A->view(), row_begin);
      if (row_begin < A->nrows && ntw == 0)
        LAUNCH(ctx, k_spmm_b2<true>, spb2_grid(A->nrows - row_begin, nb), SPB_THREADS, 0, A->view(), coef, D2C(x),
               D2C(z), D2(y), nb, row_begin, alpha, beta);
    } else if (npairs > 0 && row_begin < A->nrows) {
      // paired rows and a tail of single rows (K = [F JT; J 0]) in one launch
      const unsigned tb = spb2_grid(A->nrows - row_begin, nb);
      const unsigned grid = tb + spp_grid(npairs, nb);
      LAUNCH_B(ctx, k_spmm_k2, h2, grid, SPB_THREADS, 0, A->view(), coef, D2C(x), D2C(z), D2(y), nb, npairs,
               (int)tb, alpha, beta);
    } else if (npairs > 0) {
      LAUNCH_B(ctx, k_spmm_p2, h2, spp_grid(npairs, nb), SPB_THREADS, 0, A->view(), coef, D2C(x), D2C(z), D2(y),
               nb, npairs, alpha, beta);
    } else {
      LAUNCH_B(ctx, k_spmm_b2, h2, spb2_grid(A->nrows, nb), SPB_THREADS, 0, A->view(), coef, D2C(x), D2C(z),
               D2(y), nb, 0, alpha, beta);
    }
  } else if (batched_ok(A, nb)) {
    const int gpc = spb_gpc(ctx, A->nrows, nb);
    LAUNCH_B(ctx, k_spmm_b, A->has2 && coef, spb_grid(A->nrows, nb, gpc), SPB_THREADS, 0, A->view(), coef, x, z,
             y, nb, gpc, alpha, beta);
  } else if (nb == 1) {
    const size_t threads = (size_t)A->nrows * 8;
    LAUNCH(ctx, k_spmm<8>, cdiv(threads, 256), 256, 0, A->view(), coef, x, z, y,
           nb, alpha, beta);
  } else {
    const size_t threads = (size_t)A->nrows * nb;
    LAUNCH(ctx, k_spmm<1>, cdiv(threads, 256), 256, 0, A->view(), coef, x, z, y,
           nb, alpha, beta);
  }
}

// ===========================================================================
// context
// ===========================================================================
static void fill_tabulation(double phi[7][6], double dphi[7][6][3], double qw[7], double lam[7][3]) {
  const double s15 = std::sqrt(15.0);
  const double a1 = (6.0 - s15) / 21.0, a2 = (6.0 + s15) / 21.0;
  const double w1 = (155.0 - s15) / 1200.0, w2 = (155.0 + s15) / 1200.0;
  const double qp[7][3] = {{1. / 3, 1. / 3, 1. / 3},
                           {1 - 2 * a1, a1, a1}, {a1, 1 - 2 * a1, a1}, {a1, a1, 1 - 2 * a1},
                           {1 - 2 * a2, a2, a2}, {a2, 1 - 2 * a2, a2}, {a2, a2, 1 - 2 * a2}};
  const double w[7] = {9. / 40, w1, w1, w1, w2, w2, w2};
  for (int q = 0; q < 7; ++q) {
    const double l0 = qp[q][0], l1 = qp[q][1], l2 = qp[q][2];
    qw[q] = w[q];
    lam[q][0] = l0; lam[q][1] = l1; lam[q][2] = l2;
    phi[q][0] = l0 * (2 * l0 - 1); phi[q][1] = l1 * (2 * l1 - 1);
    phi[q][2] = l2 * (2 * l2 - 1); phi[q][3] = 4 * l1 * l2;
    phi[q][4] = 4 * l0 * l2;       phi[q][5] = 4 * l0 * l1;
    for (int a = 0; a < 6; ++a)
      for (int i = 0; i < 3; ++i) dphi[q][a][i] = 0.0;
    dphi[q][0][0] = 4 * l0 - 1; dphi[q][1][1] = 4 * l1 - 1; dphi[q][2][2] = 4 * l2 - 1;
    dphi[q][3][1] = 4 * l2; dphi[q][3][2] = 4 * l1;
    dphi[q][4][0] = 4 * l2; dphi[q][4][2] = 4 * l0;
    dphi[q][5][0] = 4 * l1; dphi[q][5][1] = 4 * l0;
  }
}

// The tuning switches are file-scope variables (read by the launch helpers above), but they BELONG to a
// context: the DNSB_* environment is read when a context is created and stored with it, and every entry
// point makes its context's set the current one (dnsb_enter).  Two contexts created under different
// switches can be used side by side in one process (the parity tests do); contexts are not thread safe.
#define DNSB_SWITCH_LIST(X) X(g_rows_per_cta) X(g_pair) X(g_tma_min_rows) X(g_gs_tma) X(g_tma_rows) X(g_tma_stages) \
  X(g_dmma) X(g_schur_tf32) X(g_schur_tc) X(g_tile) X(g_gs_pyth) X(g_schur_l2keep) X(g_tile_stages)             \
  X(g_tile_stages_f) X(g_tail_warps) X(g_pkeep) X(g_proj_t) X(g_cheb_f32) X(g_conv_colours) X(g_rowpair)         \
  X(g_graphs) X(g_dense_ctas_per_sm) X(g_tilef_ctas) X(g_tc_ctas) X(g_init_tile)
#define X(name) &name,
static int *const g_switches[] = {DNSB_SWITCH_LIST(X)};
#undef X
static void switches_store(int *sw) {
  for (const int *v : g_switches) *sw++ = *v;
}
static void switches_load(const int *sw) {
  for (int *v : g_switches) *v = *sw++;
}
static const dnsb_ctx *g_switch_owner = nullptr;
static inline cudaError_t dnsb_enter(const dnsb_ctx *ctx) {
  if (g_switch_owner != ctx) { switches_load(ctx->sw); g_switch_owner = ctx; }
  return cudaSetDevice(ctx->device);
}

extern "C" int dnsb_version(void) { return DNSB_VERSION; }

// lets each kernel use up to `bytes` of dynamic shared memory
template <class... K>
static cudaError_t smem_optin(int bytes, K *...kern) {
  for (const void *k : {(const void *)kern...})
    if (const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)) return e;
  return cudaSuccess;
}

extern "C" int dnsb_ctx_create(int device, dnsb_ctx **out) {
  if (!out) return -2;
  *out = nullptr;
  dnsb_ctx *ctx = new (std::nothrow) dnsb_ctx();
  if (!ctx) return -3;
  ctx->device = device;
  {
    static int defaults[32];
    static bool have_defaults = false;
    if (!have_defaults) { switches_store(defaults); have_defaults = true; }
    switches_load(defaults);   // the environment below is applied to the defaults, not to the last context's set
  }
  if (const char *ev = getenv("DNSB_ROWS_PER_CTA")) g_rows_per_cta = std::max(1, atoi(ev));
  if (const char *ev = getenv("DNSB_PAIR")) g_pair = atoi(ev);
  if (const char *ev = getenv("DNSB_TMA_MIN_ROWS")) g_tma_min_rows = atoi(ev);
  if (const char *ev = getenv("DNSB_GS_TMA")) g_gs_tma = atoi(ev);
  if (const char *ev = getenv("DNSB_TMA_ROWS")) g_tma_rows = std::min(SPT_ROWS, std::max(4, atoi(ev) & ~3));
  if (const char *ev = getenv("DNSB_TMA_STAGES")) g_tma_stages = std::min(SPT_MAX_STAGES, std::max(2, atoi(ev)));
  if (const char *ev = getenv("DNSB_DMMA")) g_dmma = atoi(ev);
  if (const char *ev = getenv("DNSB_SCHUR_TF32")) g_schur_tf32 = atoi(ev);
  if (const char *ev = getenv("DNSB_SCHUR_TC")) g_schur_tc = atoi(ev);
  if (const char *ev = getenv("DNSB_TILE")) g_tile = atoi(ev);
  if (const char *ev = getenv("DNSB_GS_PYTH")) g_gs_pyth = atoi(ev);
  if (const char *ev = getenv("DNSB_INIT_TILE")) g_init_tile = atoi(ev);
  if (const char *ev = getenv("DNSB_TC_CTAS")) g_tc_ctas = atoi(ev);
  if (const char *ev = getenv("DNSB_TILEF_CTAS")) g_tilef_ctas = atoi(ev);
  if (const char *ev = getenv("DNSB_PDL")) ctx->pdl = atoi(ev);
  if (const char *ev = getenv("DNSB_PDL_ONLY")) ctx->pdl_only = ev;
  if (const char *ev = getenv("DNSB_PDL_SKIP")) ctx->pdl_skip = ev;
  if (const char *ev = getenv("DNSB_SCHUR_L2KEEP")) g_schur_l2keep = atoi(ev);
  if (const char *ev = getenv("DNSB_TILE_STAGES")) g_tile_stages = std::max(2, std::min(TILE_MAX_STAGES, atoi(ev)));
  if (const char *ev = getenv("DNSB_TILE_STAGES_F")) g_tile_stages_f = std::max(2, std::min(TILE_MAX_STAGES, atoi(ev)));
  if (const char *ev = getenv("DNSB_TAIL_WARPS")) g_tail_warps = std::max(0, std::min(TILE_TAIL_WARPS_MAX, atoi(ev)));
  if (const char *ev = getenv("DNSB_PKEEP")) g_pkeep = atoi(ev);
  if (const char *ev = getenv("DNSB_PROJ_T")) g_proj_t = atoi(ev);
  if (const char *ev = getenv("DNSB_CHEB_F32")) g_cheb_f32 = atoi(ev);
  if (const char *ev = getenv("DNSB_CONV_COLOURS")) g_conv_colours = atoi(ev);
  if (const char *ev = getenv("DNSB_ROWPAIR")) g_rowpair = atoi(ev);
  if (const char *ev = getenv("DNSB_GRAPHS")) g_graphs = atoi(ev);
  if (const char *ev = getenv("DNSB_DENSE_CTAS_PER_SM")) g_dense_ctas_per_sm = std::max(1, atoi(ev));
  switches_store(ctx->sw);
  g_switch_owner = ctx;
  *out = ctx;   // returned even on failure so that the message can be read
  DNSB_CK(ctx, cudaSetDevice(device));
  cudaDeviceProp prop;
  DNSB_CK(ctx, cudaGetDeviceProperties(&prop, device));
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cc = prop.major * 10 + prop.minor;
  ctx->mem_bytes = prop.totalGlobalMem;
  DNSB_CK(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  double phi[7][6], dphi[7][6][3], qw[7], lam[7][3];
  fill_tabulation(phi, dphi, qw, lam);
  DNSB_CK(ctx, cudaMemcpyToSymbol(c_phi, phi, sizeof phi));
  DNSB_CK(ctx, cudaMemcpyToSymbol(c_dphi, dphi, sizeof dphi));
  DNSB_CK(ctx, cudaMemcpyToSymbol(c_qw, qw, sizeof qw));
  DNSB_CK(ctx, cudaMemcpyToSymbol(c_lam, lam, sizeof lam));
  // every kernel that takes more than 48 KB of dynamic shared memory, by the most it takes
  DNSB_CK(ctx, smem_optin(200 * 1024, k_mdot_b));   // (nvec+1) x 256 partial sums
  DNSB_CK(ctx, smem_optin(112 * 1024, k_gs_tma<false>, k_gs_tma<true>));
  DNSB_CK(ctx, smem_optin((int)SPT_SMEM_OPTIN, k_spmv_tma<true, SPT_AXPBY>, k_spmv_tma<false, SPT_AXPBY>,
                          k_spmv_tma<true, SPT_CHEB_INIT>, k_spmv_tma<false, SPT_CHEB_INIT>,
                          k_spmv_tma<true, SPT_CHEB_STEP>, k_spmv_tma<false, SPT_CHEB_STEP>,
                          k_spmv_tma<true, SPT_CHEB_STEP_FIRST>, k_spmv_tma<false, SPT_CHEB_STEP_FIRST>,
                          k_spmv_tma<true, SPT_CHEB_STEP_LAST>, k_spmv_tma<false, SPT_CHEB_STEP_LAST>,
                          k_spmv_tma<true, SPT_CHEB_STEP_ONLY>, k_spmv_tma<false, SPT_CHEB_STEP_ONLY>));
  DNSB_CK(ctx, smem_optin(DMM_SMEM_BYTES, k_dense_dmma_streamk));
  DNSB_CK(ctx, smem_optin(TFM_SMEM_BYTES, k_dense_tf32_streamk<1>, k_dense_tf32_streamk<2>, k_dense_tf32_streamk<3>));
  DNSB_CK(ctx, smem_optin(TC_SMEM_OPTIN, k_schur_tc));
  DNSB_CK(ctx, smem_optin(96 * 1024, k_gmres_givens));
  DNSB_CK(ctx, smem_optin(TILE_SMEM_OPTIN, k_cheb_step_tile<true, true>, k_cheb_step_tile<true, false>,
                          k_cheb_step_tile<false, true>, k_cheb_step_tile<false, false>, k_spmm_tile<true>,
                          k_spmm_tile<false>, k_cheb_init_tilef, k_cheb_step_tilef<true, true>,
                          k_cheb_step_tilef<true, false>, k_cheb_step_tilef<false, true>,
                          k_cheb_step_tilef<false, false>));
  return 0;
}

extern "C" void dnsb_ctx_destroy(dnsb_ctx *ctx) {
  if (!ctx) return;
  dnsb_enter(ctx);
  g_switch_owner = nullptr;
  delete ctx;
}

extern "C" void dnsb_live_bytes(long long *device, long long *pinned) {
  if (device) *device = g_live_bytes[0];
  if (pinned) *pinned = g_live_bytes[1];
}

extern "C" const char *dnsb_last_error(dnsb_ctx *ctx) {
  return ctx ? ctx->err.c_str() : "null context";
}

extern "C" int dnsb_device_info(dnsb_ctx *ctx, int *sm_count, size_t *mem_bytes, int *cc) {
  if (!ctx) return -2;
  if (sm_count) *sm_count = ctx->sm_count;
  if (mem_bytes) *mem_bytes = ctx->mem_bytes;
  if (cc) *cc = ctx->cc;
  return 0;
}

extern "C" int dnsb_sync(dnsb_ctx *ctx) {
  if (!ctx) return -2;
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dnsb_profile_begin(dnsb_ctx *ctx, int max_records) {
  if (!ctx) return -2;
  DNSB_CK(ctx, dnsb_enter(ctx));
  ctx->drop_recs();
  ctx->prof_cap = max_records > 0 ? (size_t)max_records : 0;
  ctx->prof = max_records > 0;
  return 0;
}

// "name count total_ms\n" per kernel, sorted by total time; returns the
// number of bytes needed (incl. the terminating 0) or < 0 on error
extern "C" int dnsb_profile_end(dnsb_ctx *ctx, char *buf, int buflen) {
  if (!ctx) return -2;
  DNSB_CK(ctx, dnsb_enter(ctx));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->prof = false;
  std::vector<std::string> names;
  std::vector<double> tot;
  std::vector<long long> cnt, work;
  for (ProfRec &r : ctx->recs) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    size_t k = 0;
    for (; k < names.size(); ++k) if (names[k] == r.name) break;
    if (k == names.size()) { names.push_back(r.name); tot.push_back(0.0); cnt.push_back(0); work.push_back(0); }
    tot[k] += ms; cnt[k] += 1; work[k] += r.work;
  }
  ctx->drop_recs();
  std::vector<size_t> order(names.size());
  for (size_t k = 0; k < order.size(); ++k) order[k] = k;
  std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return tot[a] > tot[b]; });
  std::string out;
  char line[256];
  for (size_t k : order) {
    snprintf(line, sizeof line, "%s %lld %.6f %lld\n", names[k].c_str(), cnt[k], tot[k], work[k]);
    out += line;
  }
  if (buf && buflen > 0) {
    const size_t ncopy = std::min((size_t)buflen - 1, out.size());
    memcpy(buf, out.data(), ncopy);
    buf[ncopy] = 0;
  }
  return (int)out.size() + 1;
}

extern "C" long long dnsb_launch_count(dnsb_ctx *ctx) { return ctx ? ctx->launches : -1; }
extern "C" void dnsb_launch_count_reset(dnsb_ctx *ctx) { if (ctx) ctx->launches = 0; }

// ===========================================================================
// mesh + convection
// ===========================================================================
extern "C" int dnsb_set_mesh(dnsb_ctx *ctx, int ncell, int nnodes,
                             const int32_t *cell_nodes, const double *geom,
                             int ncolours, const int32_t *cell_colour) {
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, ncell > 0 && nnodes > 0 && cell_nodes && geom && cell_colour &&
               ncolours > 0, "bad mesh arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  // counting sort of the cells by colour (stable: keeps the mesh order inside
  // a colour); verify the colouring on the way (no shared node per colour)
  std::vector<int> count(ncolours + 1, 0);
  for (int c = 0; c < ncell; ++c) {
    DNSB_REQUIRE(ctx, cell_colour[c] >= 0 && cell_colour[c] < ncolours, "colour out of range");
    count[cell_colour[c] + 1]++;
  }
  for (int k = 0; k < ncolours; ++k) count[k + 1] += count[k];
  ctx->colour_ptr = count;
  std::vector<int> pos(count.begin(), count.end() - 1);
  ctx->perm.assign(ncell, 0);
  for (int c = 0; c < ncell; ++c) ctx->perm[pos[cell_colour[c]]++] = c;
  {
    std::vector<int> stamp(nnodes, -1);
    for (int k = 0; k < ncolours; ++k)
      for (int q = ctx->colour_ptr[k]; q < ctx->colour_ptr[k + 1]; ++q) {
        const int c = ctx->perm[q];
        for (int a = 0; a < 6; ++a) {
          const int nd = cell_nodes[c * 6 + a];
          DNSB_REQUIRE(ctx, nd >= 0 && nd < nnodes, "cell node out of range");
          DNSB_REQUIRE(ctx, stamp[nd] != k, "invalid colouring: node shared within a colour");
          stamp[nd] = k;
        }
      }
  }
  std::vector<int> cn((size_t)6 * ncell);
  std::vector<double> gm((size_t)5 * ncell);
  for (int q = 0; q < ncell; ++q) {
    const int c = ctx->perm[q];
    for (int a = 0; a < 6; ++a) cn[(size_t)a * ncell + q] = cell_nodes[c * 6 + a];
    for (int a = 0; a < 5; ++a) gm[(size_t)a * ncell + q] = geom[c * 5 + a];
  }
  {
    // node -> incident (cell, local node) pairs, in ascending (permuted) cell order
    std::vector<int> ptr(nnodes + 1, 0), idx((size_t)6 * ncell);
    for (int q = 0; q < ncell; ++q)
      for (int a = 0; a < 6; ++a) ptr[cn[(size_t)a * ncell + q] + 1]++;
    for (int k = 0; k < nnodes; ++k) ptr[k + 1] += ptr[k];
    std::vector<int> fill(ptr.begin(), ptr.end() - 1);
    for (int q = 0; q < ncell; ++q)
      for (int a = 0; a < 6; ++a) idx[fill[cn[(size_t)a * ncell + q]]++] = q * 6 + a;
    DNSB_CK(ctx, ctx->n2c_ptr.upload(ptr.data(), ptr.size(), ctx->stream));
    DNSB_CK(ctx, ctx->n2c_idx.upload(idx.data(), idx.size(), ctx->stream));
  }
  DNSB_CK(ctx, ctx->cn.upload(cn.data(), cn.size(), ctx->stream));
  DNSB_CK(ctx, ctx->geom.upload(gm.data(), gm.size(), ctx->stream));
  ctx->ncell = ncell; ctx->nnodes = nnodes; ctx->ncolours = ncolours;
  {
    unsigned long long hsh = 1469598103934665603ull;   // FNV-1a
    const unsigned char *pb = reinterpret_cast<const unsigned char *>(cell_nodes);
    for (size_t k = 0; k < (size_t)6 * ncell * sizeof(int32_t); ++k) { hsh ^= pb[k]; hsh *= 1099511628211ull; }
    pb = reinterpret_cast<const unsigned char *>(geom);
    for (size_t k = 0; k < (size_t)5 * ncell * sizeof(double); ++k) { hsh ^= pb[k]; hsh *= 1099511628211ull; }
    ctx->mesh_hash = hsh;
  }
  ctx->cnnz = 0;
  return 0;
}

extern "C" int dnsb_set_conv_pattern(dnsb_ctx *ctx, const int32_t *indptr,
                                     const int32_t *indices, const int32_t *cell_slots) {
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, ctx->ncell > 0, "set the mesh first");
  DNSB_REQUIRE(ctx, indptr && indices && cell_slots, "null pattern");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int nrows = 2 * ctx->nnodes;
  const int nnz = indptr[nrows];
  const int ncell = ctx->ncell;
  std::vector<int> sl((size_t)144 * ncell);
  for (int q = 0; q < ncell; ++q) {
    const int c = ctx->perm[q];
    for (int e = 0; e < 144; ++e) {
      const int s = cell_slots[(size_t)c * 144 + e];
      DNSB_REQUIRE(ctx, s >= 0 && s < nnz, "cell slot out of range");
      sl[(size_t)e * ncell + q] = s;
    }
  }
  DNSB_CK(ctx, ctx->cindptr.upload(indptr, nrows + 1, ctx->stream));
  DNSB_CK(ctx, ctx->cindices.upload(indices, nnz, ctx->stream));
  DNSB_CK(ctx, ctx->cslots.upload(sl.data(), sl.size(), ctx->stream));
  {
    // slot -> contributions (permuted cell*144 + e), ascending cell order
    std::vector<int> sp(nnz + 1, 0), ss((size_t)144 * ncell);
    for (size_t k = 0; k < sl.size(); ++k) sp[sl[k] + 1]++;
    for (int k = 0; k < nnz; ++k) sp[k + 1] += sp[k];
    std::vector<int> fill(sp.begin(), sp.end() - 1);
    for (int q = 0; q < ncell; ++q)
      for (int e = 0; e < 144; ++e) ss[fill[sl[(size_t)e * ncell + q]]++] = q * 144 + e;
    DNSB_CK(ctx, ctx->cslot_ptr.upload(sp.data(), sp.size(), ctx->stream));
    DNSB_CK(ctx, ctx->cslot_src.upload(ss.data(), ss.size(), ctx->stream));
  }
  ctx->cnnz = nnz;
  return 0;
}

// out = sign * c(u1,u2) on device vectors: all 2*nnodes dofs (dofs == null,
// nout = 2*nnodes) or the listed dofs only; out is overwritten.
// Gather formulation by default (2 launches); DNSB_CONV_COLOURS=1 selects the
// coloured scatter (one launch per colour), which only writes full vectors.
static int convvec_dev(dnsb_ctx *ctx, const double *u1, const double *u2,
                       double *out, int nb, const int *dofs = nullptr, int nout = -1,
                       double sign = 1.0) {
  const bool same = (u2 == nullptr || u2 == u1);
  if (g_conv_colours && dofs == nullptr && sign == 1.0) {
    const size_t nfull = (size_t)2 * ctx->nnodes * nb;
    DNSB_CK(ctx, cudaMemsetAsync(out, 0, nfull * sizeof(double), ctx->stream));
    for (int k = 0; k < ctx->ncolours; ++k) {
      const int c0 = ctx->colour_ptr[k], c1 = ctx->colour_ptr[k + 1];
      if (c1 <= c0) continue;
      const size_t threads = (size_t)(c1 - c0) * nb;
      if (same)
        LAUNCH(ctx, k_convvec<true>, cdiv(threads, 128), 128, 0, c0, c1, ctx->ncell,
               ctx->cn.p, ctx->geom.p, u1, u1, out, nb);
      else
        LAUNCH(ctx, k_convvec<false>, cdiv(threads, 128), 128, 0, c0, c1, ctx->ncell,
               ctx->cn.p, ctx->geom.p, u1, u2, out, nb);
    }
    return 0;
  }
  DNSB_CK(ctx, ctx->elem.alloc((size_t)12 * ctx->ncell * nb));
  const size_t threads = (size_t)ctx->ncell * nb;
  if (same)
    LAUNCH(ctx, k_conv_elem<true>, cdiv(threads, 128), 128, 0, ctx->ncell, ctx->cn.p, ctx->geom.p,
           u1, u1, ctx->elem.p, nb);
  else
    LAUNCH(ctx, k_conv_elem<false>, cdiv(threads, 128), 128, 0, ctx->ncell, ctx->cn.p, ctx->geom.p,
           u1, u2, ctx->elem.p, nb);
  if (nout < 0) nout = 2 * ctx->nnodes;
  LAUNCH(ctx, k_conv_gather, cdiv((size_t)nout * nb, 256), 256, 0, nout, dofs,
         (const int *)ctx->n2c_ptr.p, (const int *)ctx->n2c_idx.p, (const double *)ctx->elem.p, out,
         nb, sign);
  return 0;
}

extern "C" int dnsb_convvec(dnsb_ctx *ctx, const double *u1, const double *u2,
                            double *out, int nb) {
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, ctx->ncell > 0, "set the mesh first");
  DNSB_REQUIRE(ctx, u1 && out && nb >= 1, "bad arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t nfull = (size_t)2 * ctx->nnodes * nb;
  DNSB_CK(ctx, ctx->stage_a.upload(u1, nfull, ctx->stream));
  if (u2) DNSB_CK(ctx, ctx->stage_b.upload(u2, nfull, ctx->stream));
  DNSB_CK(ctx, ctx->stage_c.alloc(nfull));
  int rc = convvec_dev(ctx, ctx->stage_a.p, u2 ? ctx->stage_b.p : nullptr,
                       ctx->stage_c.p, nb);
  if (rc) return rc;
  DNSB_CK(ctx, cudaMemcpyAsync(out, ctx->stage_c.p, nfull * sizeof(double),
                               cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// K1b on device vectors: n1, n2 (full pattern values), f3 (full vector); any of
// n1 / n2 / f3 may be null.  Gather formulation (2 launches + K1a for f3);
// DNSB_CONV_COLOURS=1 selects the coloured scatter (one launch per colour).
static int convmats_dev(dnsb_ctx *ctx, const double *u0, double *n1, double *n2, double *f3) {
  const size_t nfull = (size_t)2 * ctx->nnodes, nnz = ctx->cnnz;
  if (g_conv_colours) {
    if (n1) DNSB_CK(ctx, cudaMemsetAsync(n1, 0, nnz * sizeof(double), ctx->stream));
    if (n2) DNSB_CK(ctx, cudaMemsetAsync(n2, 0, nnz * sizeof(double), ctx->stream));
    if (f3) DNSB_CK(ctx, cudaMemsetAsync(f3, 0, nfull * sizeof(double), ctx->stream));
    for (int k = 0; k < ctx->ncolours; ++k) {
      const int c0 = ctx->colour_ptr[k], c1 = ctx->colour_ptr[k + 1];
      if (c1 <= c0) continue;
      const size_t threads = (size_t)(c1 - c0) * 6;
      LAUNCH(ctx, k_convmats, cdiv(threads, 128), 128, 0, c0, c1, ctx->ncell, ctx->cn.p, ctx->geom.p,
             ctx->cslots.p, u0, n1, n2, f3);
    }
    return 0;
  }
  DNSB_CK(ctx, ctx->en1.alloc((size_t)36 * ctx->ncell));
  DNSB_CK(ctx, ctx->en2.alloc((size_t)144 * ctx->ncell));
  LAUNCH(ctx, k_convmats_elem, cdiv((size_t)ctx->ncell, CME_CELLS), 6 * CME_CELLS, 0, ctx->ncell, ctx->cn.p,
         ctx->geom.p, u0, ctx->en1.p, ctx->en2.p);
  LAUNCH(ctx, k_convmats_gather, cdiv(nnz, 256), 256, 0, (int)nnz, ctx->ncell, (const int *)ctx->cslot_ptr.p,
         (const int *)ctx->cslot_src.p, (const double *)ctx->en1.p, (const double *)ctx->en2.p, n1, n2);
  if (f3) return convvec_dev(ctx, u0, nullptr, f3, 1);
  return 0;
}

// slot -> contributions for a per-cell element array of `per` entries: the caller gives, for every
// HOST cell, the CSR slot of each of its `per` entries; the lists are built in device cell order
static int slot_lists(dnsb_ctx *ctx, int per, int nslots, const int32_t *cell_slots, DBuf<int> &sptr,
                      DBuf<int> &ssrc) {
  const int ncell = ctx->ncell;
  std::vector<int> sp(nslots + 1, 0), ss((size_t)per * ncell);
  for (size_t k = 0; k < (size_t)per * ncell; ++k) {
    DNSB_REQUIRE(ctx, cell_slots[k] >= 0 && cell_slots[k] < nslots, "cell slot out of range");
    sp[cell_slots[k] + 1]++;
  }
  for (int k = 0; k < nslots; ++k) sp[k + 1] += sp[k];
  std::vector<int> fill(sp.begin(), sp.end() - 1);
  for (int q = 0; q < ncell; ++q) {
    const int c = ctx->perm[q];
    for (int e = 0; e < per; ++e) ss[fill[cell_slots[(size_t)c * per + e]]++] = q * per + e;
  }
  DNSB_CK(ctx, sptr.upload(sp.data(), sp.size(), ctx->stream));
  DNSB_CK(ctx, ssrc.upload(ss.data(), ss.size(), ctx->stream));
  return 0;
}

extern "C" int dnsb_assemble_stokes(dnsb_ctx *ctx, double nu, int symgrad, int jnnz,
                                    const int32_t *jslots, int mpnnz, const int32_t *mpslots,
                                    double *m_vals, double *a_vals, double *j_vals,
                                    double *mp_vals) {
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, ctx->ncell > 0 && ctx->cnnz > 0, "set mesh and pattern first");
  DNSB_REQUIRE(ctx, m_vals && a_vals, "null output");
  DNSB_REQUIRE(ctx, (!j_vals || (jslots && jnnz > 0)) && (!mp_vals || (mpslots && mpnnz > 0)),
               "slot lists of J / MP missing");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int ncell = ctx->ncell;
  const size_t nnz = ctx->cnnz;
  DBuf<double> ej, emp, dm, da, dj, dmp;
  DBuf<int> jp, js, pp, ps;
  DNSB_CK(ctx, ctx->en1.alloc((size_t)36 * ncell));
  DNSB_CK(ctx, ctx->en2.alloc((size_t)144 * ncell));
  DNSB_CK(ctx, dm.alloc(nnz));
  DNSB_CK(ctx, da.alloc(nnz));
  if (j_vals) { DNSB_CK(ctx, ej.alloc((size_t)36 * ncell)); DNSB_CK(ctx, dj.alloc(jnnz)); }
  if (mp_vals) { DNSB_CK(ctx, emp.alloc((size_t)9 * ncell)); DNSB_CK(ctx, dmp.alloc(mpnnz)); }
  if (j_vals) { int rc = slot_lists(ctx, 36, jnnz, jslots, jp, js); if (rc) return rc; }
  if (mp_vals) { int rc = slot_lists(ctx, 9, mpnnz, mpslots, pp, ps); if (rc) return rc; }
  LAUNCH(ctx, k_stokes_elem, cdiv((size_t)ncell, CME_CELLS), 6 * CME_CELLS, 0, ncell,
         (const double *)ctx->geom.p, nu, symgrad, ctx->en1.p, ctx->en2.p, j_vals ? ej.p : (double *)nullptr,
         mp_vals ? emp.p : (double *)nullptr);
  LAUNCH(ctx, k_convmats_gather, cdiv(nnz, 256), 256, 0, (int)nnz, ncell, (const int *)ctx->cslot_ptr.p,
         (const int *)ctx->cslot_src.p, (const double *)ctx->en1.p, (const double *)ctx->en2.p, dm.p, da.p);
  if (j_vals)
    LAUNCH(ctx, k_slot_gather, cdiv((size_t)jnnz, 256), 256, 0, jnnz, (const int *)jp.p, (const int *)js.p,
           (const double *)ej.p, dj.p);
  if (mp_vals)
    LAUNCH(ctx, k_slot_gather, cdiv((size_t)mpnnz, 256), 256, 0, mpnnz, (const int *)pp.p, (const int *)ps.p,
           (const double *)emp.p, dmp.p);
  DNSB_CK(ctx, cudaMemcpyAsync(m_vals, dm.p, nnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaMemcpyAsync(a_vals, da.p, nnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (j_vals)
    DNSB_CK(ctx, cudaMemcpyAsync(j_vals, dj.p, (size_t)jnnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (mp_vals)
    DNSB_CK(ctx, cudaMemcpyAsync(mp_vals, dmp.p, (size_t)mpnnz * sizeof(double), cudaMemcpyDeviceToHost,
                                 ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int dnsb_convmats(dnsb_ctx *ctx, const double *u0, double *n1_data,
                             double *n2_data, double *f3) {
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, ctx->ncell > 0 && ctx->cnnz > 0, "set mesh and pattern first");
  DNSB_REQUIRE(ctx, u0 != nullptr, "null u0");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t nfull = (size_t)2 * ctx->nnodes;
  const size_t nnz = ctx->cnnz;
  DNSB_CK(ctx, ctx->stage_a.upload(u0, nfull, ctx->stream));
  DNSB_CK(ctx, ctx->stage_b.alloc(nnz));
  DNSB_CK(ctx, ctx->stage_c.alloc(nnz));
  DNSB_CK(ctx, ctx->stage_d.alloc(nfull));
  {
    int rc = convmats_dev(ctx, ctx->stage_a.p, n1_data ? ctx->stage_b.p : nullptr, n2_data ? ctx->stage_c.p : nullptr,
                          f3 ? ctx->stage_d.p : nullptr);
    if (rc) return rc;
  }
  if (n1_data) DNSB_CK(ctx, cudaMemcpyAsync(n1_data, ctx->stage_b.p, nnz * sizeof(double),
                                            cudaMemcpyDeviceToHost, ctx->stream));
  if (n2_data) DNSB_CK(ctx, cudaMemcpyAsync(n2_data, ctx->stage_c.p, nnz * sizeof(double),
                                            cudaMemcpyDeviceToHost, ctx->stream));
  if (f3) DNSB_CK(ctx, cudaMemcpyAsync(f3, ctx->stage_d.p, nfull * sizeof(double),
                                       cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// ===========================================================================
// CSR API
// ===========================================================================
extern "C" int dnsb_csr_create(dnsb_ctx *ctx, int nrows, int ncols,
                               const int32_t *indptr, const int32_t *indices,
                               const double *vals1, const double *vals2,
                               dnsb_csr **out) {
  if (out) *out = nullptr;
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, out != nullptr, "bad csr args");
  DNSB_CK(ctx, dnsb_enter(ctx));
  std::unique_ptr<dnsb_csr> m;
  int rc = csr_build(ctx, nrows, ncols, indptr, indices, vals1, vals2, m);
  if (rc) return rc;
  *out = m.release();
  return 0;
}

extern "C" void dnsb_csr_destroy(dnsb_csr *mat) {
  if (!mat) return;
  dnsb_enter(mat->ctx);
  delete mat;
}

extern "C" int dnsb_spmm_dev(dnsb_csr *mat, const double *coef_dev,
                             const double *x_dev, double *y_dev, int nb,
                             double alpha, double beta) {
  if (!mat) return -2;
  dnsb_ctx *ctx = mat->ctx;
  DNSB_REQUIRE(ctx, x_dev && y_dev && nb >= 1, "bad arguments");
  DNSB_REQUIRE(ctx, !(mat->has2 && coef_dev == nullptr), "matrix has a second value array: coef required");
  DNSB_CK(ctx, dnsb_enter(ctx));
  spmm_dev(ctx, mat, coef_dev, x_dev, y_dev, y_dev, nb, alpha, beta);
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int dnsb_spmm(dnsb_csr *mat, const double *coef, const double *x,
                         double *y, int nb, double alpha, double beta) {
  if (!mat) return -2;
  dnsb_ctx *ctx = mat->ctx;
  DNSB_REQUIRE(ctx, x && y && nb >= 1, "bad arguments");
  DNSB_REQUIRE(ctx, !(mat->has2 && coef == nullptr), "matrix has a second value array: coef required");
  DNSB_CK(ctx, dnsb_enter(ctx));
  DNSB_CK(ctx, ctx->stage_a.upload(x, (size_t)mat->ncols * nb, ctx->stream));
  if (beta != 0.0)
    DNSB_CK(ctx, ctx->stage_b.upload(y, (size_t)mat->nrows * nb, ctx->stream));
  else
    DNSB_CK(ctx, ctx->stage_b.alloc((size_t)mat->nrows * nb));
  if (coef) DNSB_CK(ctx, ctx->stage_c.upload(coef, nb, ctx->stream));
  spmm_dev(ctx, mat, coef ? ctx->stage_c.p : nullptr, ctx->stage_a.p, ctx->stage_b.p,
           ctx->stage_b.p, nb, alpha, beta);
  DNSB_CK(ctx, cudaMemcpyAsync(y, ctx->stage_b.p, (size_t)mat->nrows * nb * sizeof(double),
                               cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// ===========================================================================
// saddle-point solver
// ===========================================================================
// one level of a multigrid hierarchy (pressure/Schur block or velocity block)
enum { MG_MULTI = 0, MG_DENSE = 1, MG_SMOOTH = 2 };
struct MgLevel {
  dnsb_csr *A = nullptr, *P = nullptr, *R = nullptr;
  const double *coef = nullptr;   // per-member coefficient of A.v2 (level 0 of the velocity block)
  int n = 0, nsmooth = 1, kind = MG_MULTI;
  double lmin = 0, lmax = 0;
  DBuf<double> dinv_dense;   // n*n (MG_DENSE)
  DBuf<double> gpart;        // split-K partial sums of the dense solve
  DBuf<float> dinv_f32, x_f32;   // fp32 copies for the optional TF32 variant (DNSB_SCHUR_TF32)
  int ldf = 0;
  TcPlan tc;                     // tcgen05 variant (DNSB_SCHUR_TC): tensor maps, split-K shape
  DBuf<float> xt, tcpart;        // K-major fp32 copy of X (NP x ldx), split-K partial tiles
  DBuf<double> dinv_own;     // n*nb Jacobi (owned)
  const double *dinv = nullptr;
  DBuf<double> b, x, r, d0, d1, t;   // n*nb work vectors
};

struct dnsb_solver {
  dnsb_ctx *ctx = nullptr;
  int nv = 0, np = 0, ntot = 0, nb = 1, mr = 30, kF = 3;
  double lmin = 0, lmax = 0;
  dnsb_csr *F = nullptr, *J = nullptr, *JT = nullptr;
  std::unique_ptr<dnsb_csr> K;   // [F JT; J 0]
  DBuf<double> coef;       // nb (device copy)
  bool has_coef = false;
  DBuf<double> dinv;       // nv*nb
  DBuf<int> diagpos;
  DBuf<double> Vb, Zb, w;  // Krylov bases
  DBuf<double> cres, cd0, cd1;   // Chebyshev work (nv*nb)
  DBuf<float> cf_res, cf_d0, cf_d1, cf_z, cf_dinv;   // the same in fp32 (DNSB_CHEB_F32, tile path)
  DBuf<double> partial, partial2, red;
  RedCfg rc;
  // GMRES scalars
  DBuf<double> gR, gcs, gsn, gg, gh, gh2, ginvh, gbnorm, gresid;
  DBuf<int> gdone, gits, gittot, gflags;
  DBuf<double> grelmax;
  GmresState gs;
  PinnedBuf<int> h_flags;
  std::vector<std::unique_ptr<MgLevel>> levels;    // Schur (pressure) hierarchy
  std::vector<std::unique_ptr<MgLevel>> vlevels;   // velocity hierarchy; [0] = F itself
  DBuf<double> mp_dinv, mp_scale;
  bool has_mass = false;
  // least-squares-commutator Schur approximation (Stokes / Oseen / Newton)
  DBuf<double> lsc_dinv, lsc_t1, lsc_t2, lsc_p1, lsc_p2;
  bool has_lsc = false;
  int expect_its = 0;
  // user-facing staging
  DBuf<double> sb, sx;
  // CUDA graphs of the Arnoldi steps (one per column j), valid for one tol
  std::vector<cudaGraphExec_t> igraph;
  std::vector<int> igraph_launches;
  std::vector<int> igraph_seen;   // how often column j ran since the graphs were dropped
  int prec_diag = 0;   // 1: block-DIAGONAL, symmetric positive definite form of the preconditioner (MINRES)
  DBuf<double> zero_p;
  double igraph_tol = -1.0;
  // Pythagorean norm in the Arnoldi step: only for solves that are expected to be SHORT (the
  // previous solve of this solver took <= 8 iterations: the time loop with recycled guesses).
  // Classical Gram-Schmidt loses orthogonality as a long solve converges, and then |h|^2 is no
  // measure of |V h|^2 any more (a 25-iteration solve from a zero guess ended at 1e-8 instead of
  // 1e-12); the graphs of a solver are captured for one variant and dropped when it changes
  bool use_pyth = false, igraph_pyth = false;
  long long stat_iters = 0, stat_solves = 0, stat_launched = 0;
  long long stat_unconverged = 0;   // solves that stopped at maxit above tol
  ~dnsb_solver() {
    cudaStreamSynchronize(ctx->stream);   // no buffer is freed under a running kernel
    for (cudaGraphExec_t g : igraph) if (g) cudaGraphExecDestroy(g);
  }
};

static void solver_drop_graphs(dnsb_solver *s);

static int find_diagpos(dnsb_ctx *ctx, const dnsb_csr *A, std::vector<int> &dp) {
  dp.assign(A->nrows, -1);
  for (int i = 0; i < A->nrows; ++i) {
    for (int k = A->h_indptr[i]; k < A->h_indptr[i + 1]; ++k)
      if (A->h_indices[k] == i) { dp[i] = k; break; }
    DNSB_REQUIRE(ctx, dp[i] >= 0, "matrix has a structurally zero diagonal entry");
  }
  return 0;
}

extern "C" int dnsb_solver_create(dnsb_ctx *ctx, dnsb_csr *fmat, dnsb_csr *jmat,
                                  dnsb_csr *jtmat, const double *coef, int nb,
                                  int restart, int cheb_steps, double lmin,
                                  double lmax, dnsb_solver **out) {
  if (out) *out = nullptr;
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, fmat && jmat && jtmat && out, "null matrices");
  DNSB_REQUIRE(ctx, nb >= 1 && nb <= 256, "nb must be in 1..256");
  DNSB_REQUIRE(ctx, restart >= 2 && restart <= 400, "restart must be in 2..400");
  DNSB_REQUIRE(ctx, cheb_steps >= 1, "cheb_steps >= 1");
  DNSB_REQUIRE(ctx, lmax > lmin && lmin > 0, "need 0 < lmin < lmax");
  const int nv = fmat->nrows, np = jmat->nrows;
  DNSB_REQUIRE(ctx, fmat->ncols == nv && jmat->ncols == nv && jtmat->nrows == nv &&
               jtmat->ncols == np, "inconsistent block shapes");
  DNSB_REQUIRE(ctx, !(fmat->has2 && !coef), "fmat has two value arrays: coef required");
  DNSB_CK(ctx, dnsb_enter(ctx));
  std::unique_ptr<dnsb_solver> s(new (std::nothrow) dnsb_solver());
  DNSB_REQUIRE(ctx, s != nullptr, "out of host memory");
  s->ctx = ctx; s->nv = nv; s->np = np; s->ntot = nv + np; s->nb = nb;
  s->mr = restart; s->kF = cheb_steps; s->lmin = lmin; s->lmax = lmax;
  s->F = fmat; s->J = jmat; s->JT = jtmat;
  // ---- block matrix K = [F JT; J 0] on the host, then upload -------------
  {
    const int ntot = s->ntot;
    std::vector<int> ip(ntot + 1, 0), ix;
    std::vector<double> a1, a2;
    const size_t nnz = (size_t)fmat->nnz + jtmat->nnz + jmat->nnz;
    ix.reserve(nnz); a1.reserve(nnz);
    if (fmat->has2) a2.reserve(nnz);
    for (int i = 0; i < nv; ++i) {
      for (int k = fmat->h_indptr[i]; k < fmat->h_indptr[i + 1]; ++k) {
        ix.push_back(fmat->h_indices[k]);
        a1.push_back(fmat->h_v1[k]);
        if (fmat->has2) a2.push_back(fmat->h_v2[k]);
      }
      for (int k = jtmat->h_indptr[i]; k < jtmat->h_indptr[i + 1]; ++k) {
        ix.push_back(nv + jtmat->h_indices[k]);
        a1.push_back(jtmat->h_v1[k]);
        if (fmat->has2) a2.push_back(0.0);
      }
      ip[i + 1] = (int)ix.size();
    }
    for (int j = 0; j < np; ++j) {
      for (int k = jmat->h_indptr[j]; k < jmat->h_indptr[j + 1]; ++k) {
        ix.push_back(jmat->h_indices[k]);
        a1.push_back(jmat->h_v1[k]);
        if (fmat->has2) a2.push_back(0.0);
      }
      ip[nv + j + 1] = (int)ix.size();
    }
    int rc = csr_build(ctx, ntot, ntot, ip.data(), ix.data(), a1.data(),
                       fmat->has2 ? a2.data() : nullptr, s->K);
    if (rc) return rc;
    if (nb == TILE_NB && coef) { int rct = tile_setup(ctx, s->K.get()); if (rct) return rct; }
    // the block matrix is only needed on the device
    std::vector<int>().swap(s->K->h_indptr); std::vector<int>().swap(s->K->h_indices);
    std::vector<double>().swap(s->K->h_v1); std::vector<double>().swap(s->K->h_v2);
  }
  if (coef) {
    DNSB_CK(ctx, s->coef.upload(coef, nb, ctx->stream));
    s->has_coef = true;
  }
  if (nb == TILE_NB && coef && !fmat->tile.ok) { int rc = tile_setup(ctx, fmat); if (rc) return rc; }
  const bool want_f32 = g_cheb_f32 && nb == TILE_NB && coef && fmat->tile.ok;
  if (want_f32 && g_init_tile && !jtmat->tile.ok) { int rc = tile_setup(ctx, jtmat, true); if (rc) return rc; }
  std::vector<int> dp;
  { int rc = find_diagpos(ctx, fmat, dp); if (rc) return rc; }
  DNSB_CK(ctx, s->diagpos.upload(dp.data(), dp.size(), ctx->stream));
  const size_t nvb = (size_t)nv * nb, ntb = (size_t)s->ntot * nb;
  DNSB_CK(ctx, s->dinv.alloc(nvb));
  LAUNCH(ctx, k_diag_inv, cdiv(nvb, 256), 256, 0, fmat->view(), s->diagpos.p,
         s->has_coef ? s->coef.p : nullptr, s->dinv.p, nb);
  if (want_f32) {
    DNSB_CK(ctx, s->cf_res.alloc(nvb)); DNSB_CK(ctx, s->cf_d0.alloc(nvb)); DNSB_CK(ctx, s->cf_d1.alloc(nvb));
    DNSB_CK(ctx, s->cf_z.alloc(nvb)); DNSB_CK(ctx, s->cf_dinv.alloc(nvb));
    LAUNCH(ctx, k_f64_to_f32, cdiv(nvb, 256), 256, 0, (const double *)s->dinv.p, s->cf_dinv.p, (size_t)1, nvb, nvb);
  }
  {
    std::unique_ptr<MgLevel> V0(new (std::nothrow) MgLevel());
    DNSB_REQUIRE(ctx, V0 != nullptr, "out of host memory");
    V0->A = fmat; V0->coef = s->has_coef ? s->coef.p : nullptr;
    V0->n = nv; V0->nsmooth = s->kF; V0->kind = MG_SMOOTH;
    V0->lmin = lmin; V0->lmax = lmax; V0->dinv = s->dinv.p;
    DNSB_CK(ctx, V0->b.alloc(nvb)); DNSB_CK(ctx, V0->r.alloc(nvb));
    DNSB_CK(ctx, V0->d0.alloc(nvb)); DNSB_CK(ctx, V0->d1.alloc(nvb));
    DNSB_CK(ctx, V0->t.alloc(nvb));
    s->vlevels.push_back(std::move(V0));
  }
  DNSB_CK(ctx, s->Vb.alloc(ntb * (s->mr + 1)));
  DNSB_CK(ctx, s->Zb.alloc(ntb * s->mr));
  DNSB_CK(ctx, s->w.alloc(ntb));
  DNSB_CK(ctx, s->cres.alloc(nvb));
  DNSB_CK(ctx, s->cd0.alloc(nvb));
  DNSB_CK(ctx, s->cd1.alloc(nvb));
  s->rc = red_cfg(ctx, s->ntot, nb);
  DNSB_REQUIRE(ctx, (size_t)(s->mr + 2) * s->rc.threads * sizeof(double) <= 200 * 1024,
               "restart too large for this batch width (Gram-Schmidt shared memory)");
  DNSB_CK(ctx, s->partial.alloc((size_t)s->rc.nblocks * (s->mr + 2) * nb));
  DNSB_CK(ctx, s->partial2.alloc((size_t)s->rc.nblocks * nb));
  DNSB_CK(ctx, s->red.alloc(nb));
  const int mr = s->mr;
  DNSB_CK(ctx, s->gR.alloc((size_t)(mr + 1) * mr * nb));
  DNSB_CK(ctx, s->gcs.alloc((size_t)mr * nb));
  DNSB_CK(ctx, s->gsn.alloc((size_t)mr * nb));
  DNSB_CK(ctx, s->gg.alloc((size_t)(mr + 1) * nb));
  DNSB_CK(ctx, s->gh.alloc((size_t)(mr + 2) * nb));
  DNSB_CK(ctx, s->gh2.alloc((size_t)(mr + 2) * nb));
  DNSB_CK(ctx, s->ginvh.alloc(nb));
  DNSB_CK(ctx, s->gbnorm.alloc(nb));
  DNSB_CK(ctx, s->gresid.alloc(nb));
  DNSB_CK(ctx, s->gdone.alloc(nb));
  DNSB_CK(ctx, s->gits.alloc(nb));
  DNSB_CK(ctx, s->gittot.alloc(nb));
  DNSB_CK(ctx, s->gflags.alloc(4));
  DNSB_CK(ctx, s->grelmax.alloc(nb));
  DNSB_CK(ctx, s->grelmax.zero(ctx->stream));
  s->gs.R = s->gR.p; s->gs.cs = s->gcs.p; s->gs.sn = s->gsn.p; s->gs.g = s->gg.p;
  s->gs.h = s->gh.p; s->gs.invh = s->ginvh.p; s->gs.bnorm = s->gbnorm.p;
  s->gs.resid = s->gresid.p; s->gs.done = s->gdone.p; s->gs.its = s->gits.p;
  s->gs.ittot = s->gittot.p; s->gs.flags = s->gflags.p; s->gs.relmax = s->grelmax.p; s->gs.mr = mr;
  DNSB_CK(ctx, s->h_flags.alloc(4));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  *out = s.release();
  return 0;
}

// stream-K shape of the dense solve: `g_dense_ctas_per_sm` CTAs per SM, each
// with the same number of (row tile, k step) units
static void dense_split(dnsb_ctx *ctx, int n, int nb, int *tn, DenseSplit *sp) {
  *tn = nb <= 16 ? 16 : (nb <= 32 ? 32 : 64);
  const int rt = cdiv(n, DGK_TM);
  sp->ksteps = cdiv(n, DGK_TK);
  const long units = (long)rt * sp->ksteps;
  long P = std::min<long>(units, (long)g_dense_ctas_per_sm * ctx->sm_count);
  sp->upc = (int)((units + P - 1) / P);
  sp->nctas = (int)((units + sp->upc - 1) / sp->upc);
  sp->maxseg = 2 + sp->upc / sp->ksteps;
}

// ---- tcgen05 dense Schur block: tensor maps + split-K shape ------------------
typedef CUresult (*dnsb_encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                         const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                         const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static dnsb_encode_tiled_fn tc_encode_fn() {
  static dnsb_encode_tiled_fn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (dnsb_encode_tiled_fn)p;
  }
  return fn;
}
// a 2-D fp32 tensor (rows x cols, leading dimension ld floats) seen by TMA in boxes of
// box_rows x TC_BK with the 128-byte swizzle the UMMA descriptors expect; out-of-range = 0
static bool tc_map_2d(CUtensorMap *map, const float *base, int rows, int cols, int ld, int box_rows) {
  dnsb_encode_tiled_fn enc = tc_encode_fn();
  if (!enc) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
  const cuuint32_t box[2] = {TC_BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)base, gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// needs L->dinv_f32 (n x ldf); returns cudaSuccess with tc.ok = false when the block does not qualify
static cudaError_t tc_setup(dnsb_ctx *ctx, MgLevel *L, int n, int nb) {
  TcPlan &p = L->tc;
  p.ok = false;
  if (ctx->cc < 100 || nb < 8 || nb > 256 || n < TC_BM) return cudaSuccess;   // nb < 8: k_dense_gemv (fp64, D-bandwidth bound)
  p.np_ = (nb + 15) & ~15;
  p.kblocks = (n + TC_BK - 1) / TC_BK;
  p.mtiles = (n + TC_BM - 1) / TC_BM;
  const int per_sm = std::max(1, std::min(2, g_tc_ctas));   // resident CTAs per SM the split-K grid is sized for
  p.splits = std::max(1, std::min(p.kblocks, per_sm * ctx->sm_count / p.mtiles));
  p.kb_per_split = (p.kblocks + p.splits - 1) / p.splits;
  p.splits = (p.kblocks + p.kb_per_split - 1) / p.kb_per_split;
  const size_t a_bytes = (size_t)TC_BM * TC_BK * 4;
  const size_t b_bytes = (((size_t)p.np_ * TC_BK * 4) + 1023) & ~(size_t)1023;
  p.stages = (int)std::min<size_t>(TC_MAX_STAGES, ((size_t)TC_SMEM_OPTIN / per_sm - 1024) / (a_bytes + b_bytes));
  if (p.stages < 2) return cudaSuccess;
  p.smem = (size_t)p.stages * (a_bytes + b_bytes) + 1024;
  p.ldx = (n + 3) & ~3;
  cudaError_t e;
  if ((e = L->xt.alloc((size_t)p.np_ * p.ldx)) != cudaSuccess) return e;
  if ((e = L->xt.zero(ctx->stream)) != cudaSuccess) return e;
  if ((e = L->tcpart.alloc((size_t)p.splits * p.mtiles * TC_BM * p.np_)) != cudaSuccess) return e;
  // D: TF32-rounded fp32 copy in packed, pre-swizzled 128 x 32 tiles
  if ((e = L->dinv_f32.alloc((size_t)p.mtiles * p.kblocks * TC_BM * TC_BK)) != cudaSuccess) return e;
  LAUNCH(ctx, k_tc_pack_d, cdiv(L->dinv_f32.n, 256), 256, 0, (const double *)L->dinv_dense.p, L->dinv_f32.p, n,
         p.mtiles, p.kblocks);
  p.ok = tc_map_2d(&p.mapB, L->xt.p, p.np_, n, p.ldx, p.np_);
  return cudaSuccess;
}

extern "C" void dnsb_solver_destroy(dnsb_solver *s) {
  if (!s) return;
  dnsb_enter(s->ctx);
  delete s;
}

// append a level to the pressure (block 0) or velocity (block 1) hierarchy
static int solver_add_level(dnsb_solver *s, int block, dnsb_csr *amat, dnsb_csr *pmat,
                            dnsb_csr *rmat, int nsmooth, double lmin, double lmax,
                            const double *dense_inv) {
  dnsb_ctx *ctx = s->ctx;
  DNSB_CK(ctx, dnsb_enter(ctx));
  std::vector<std::unique_ptr<MgLevel>> &lv = block == 0 ? s->levels : s->vlevels;
  solver_drop_graphs(s);   // the preconditioner changes: captured launch sequences are stale
  int nexpect;
  if (lv.empty()) {
    DNSB_REQUIRE(ctx, block == 0, "velocity level 0 is the matrix F itself");
    nexpect = s->np;
  } else {
    const MgLevel *up = lv.back().get();
    DNSB_REQUIRE(ctx, up->kind == MG_MULTI && up->P, "previous level is terminal");
    nexpect = up->P->ncols;
  }
  std::unique_ptr<MgLevel> L(new (std::nothrow) MgLevel());
  DNSB_REQUIRE(ctx, L != nullptr, "out of host memory");
  L->n = nexpect;
  if (dense_inv) {
    L->kind = MG_DENSE;
    DNSB_CK(ctx, L->dinv_dense.upload(dense_inv, (size_t)nexpect * nexpect, ctx->stream));
    if (s->nb > 8) {
      int tn;
      DenseSplit sp;
      dense_split(ctx, nexpect, s->nb, &tn, &sp);
      DNSB_CK(ctx, L->gpart.alloc((size_t)sp.nctas * sp.maxseg * DGK_TM * s->nb));
      if (g_schur_tf32 && s->nb % 4 == 0) {
        L->ldf = (nexpect + 3) & ~3;
        DNSB_CK(ctx, L->dinv_f32.alloc((size_t)nexpect * L->ldf));
        DNSB_CK(ctx, L->x_f32.alloc((size_t)nexpect * s->nb));
        LAUNCH(ctx, k_f64_to_f32, cdiv((size_t)nexpect * L->ldf, 256), 256, 0, (const double *)L->dinv_dense.p,
               L->dinv_f32.p, (size_t)nexpect, (size_t)nexpect, (size_t)L->ldf);
      }
    }
    if (g_schur_tc && !g_schur_tf32) {
      DNSB_CK(ctx, tc_setup(ctx, L.get(), nexpect, s->nb));
      if (!L->tc.ok) {   // block does not qualify: the fp64 kernels serve it
        DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
        L->dinv_f32.release(); L->xt.release(); L->tcpart.release();
      }
    }
  } else {
    bool ok = amat && amat->nrows == nexpect && amat->ncols == nexpect && lmax > lmin &&
              lmin > 0 && nsmooth >= 1 && !amat->has2;
    if (ok && (pmat || rmat))
      ok = pmat && rmat && pmat->nrows == nexpect && rmat->ncols == nexpect &&
           rmat->nrows == pmat->ncols;
    DNSB_REQUIRE(ctx, ok, "inconsistent multigrid level");
    L->kind = pmat ? MG_MULTI : MG_SMOOTH;
    L->A = amat; L->P = pmat; L->R = rmat;
    L->nsmooth = nsmooth; L->lmin = lmin; L->lmax = lmax;
    std::vector<int> dp;
    if (find_diagpos(ctx, amat, dp)) return -2;
    {
      DBuf<int> dpd;
      DNSB_CK(ctx, dpd.upload(dp.data(), dp.size(), ctx->stream));
      const size_t nn = (size_t)nexpect * s->nb;
      DNSB_CK(ctx, L->dinv_own.alloc(nn));
      LAUNCH(ctx, k_diag_inv, cdiv(nn, 256), 256, 0, amat->view(), dpd.p,
             (const double *)nullptr, L->dinv_own.p, s->nb);
      cudaStreamSynchronize(ctx->stream);
    }
    L->dinv = L->dinv_own.p;
  }
  const size_t nn = (size_t)L->n * s->nb;
  DNSB_CK(ctx, L->b.alloc(nn)); DNSB_CK(ctx, L->x.alloc(nn)); DNSB_CK(ctx, L->r.alloc(nn));
  DNSB_CK(ctx, L->d0.alloc(nn)); DNSB_CK(ctx, L->d1.alloc(nn)); DNSB_CK(ctx, L->t.alloc(nn));
  lv.push_back(std::move(L));
  return 0;
}

extern "C" int dnsb_solver_add_schur_level(dnsb_solver *s, dnsb_csr *amat,
                                           dnsb_csr *pmat, dnsb_csr *rmat,
                                           int nsmooth, double lmin, double lmax,
                                           const double *dense_inv) {
  if (!s) return -2;
  return solver_add_level(s, 0, amat, pmat, rmat, nsmooth, lmin, lmax, dense_inv);
}

extern "C" int dnsb_solver_set_velocity_transfer(dnsb_solver *s, dnsb_csr *pmat,
                                                 dnsb_csr *rmat) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, pmat && rmat && pmat->nrows == s->nv && rmat->ncols == s->nv &&
               rmat->nrows == pmat->ncols, "inconsistent velocity transfer operators");
  DNSB_REQUIRE(ctx, s->vlevels.size() == 1, "velocity hierarchy already built");
  solver_drop_graphs(s);
  s->vlevels[0]->P = pmat; s->vlevels[0]->R = rmat;
  s->vlevels[0]->kind = MG_MULTI;
  return 0;
}

extern "C" int dnsb_solver_add_velocity_level(dnsb_solver *s, dnsb_csr *amat,
                                              dnsb_csr *pmat, dnsb_csr *rmat,
                                              int nsmooth, double lmin, double lmax,
                                              const double *dense_inv) {
  if (!s) return -2;
  return solver_add_level(s, 1, amat, pmat, rmat, nsmooth, lmin, lmax, dense_inv);
}

extern "C" int dnsb_solver_set_schur_mass(dnsb_solver *s, const double *mp_dinv,
                                          const double *mp_scale) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, mp_dinv && mp_scale, "null arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  DNSB_CK(ctx, s->mp_dinv.upload(mp_dinv, s->np, ctx->stream));
  DNSB_CK(ctx, s->mp_scale.upload(mp_scale, s->nb, ctx->stream));
  s->has_mass = true;
  solver_drop_graphs(s);
  return 0;
}

extern "C" int dnsb_solver_set_schur_lsc(dnsb_solver *s, const double *du_inv) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, du_inv != nullptr, "null argument");
  DNSB_REQUIRE(ctx, !s->levels.empty(), "add the levels of L = J Du^-1 JT first");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t nvb = (size_t)s->nv * s->nb, npb = (size_t)s->np * s->nb;
  DNSB_CK(ctx, s->lsc_dinv.upload(du_inv, s->nv, ctx->stream));
  DNSB_CK(ctx, s->lsc_t1.alloc(nvb)); DNSB_CK(ctx, s->lsc_t2.alloc(nvb));
  DNSB_CK(ctx, s->lsc_p1.alloc(npb)); DNSB_CK(ctx, s->lsc_p2.alloc(npb));
  s->has_lsc = true;
  solver_drop_graphs(s);
  return 0;
}

// dense coarse solve  y = alpha*(Dinv x [+ scale_m*mp_dinv*x])
static int dense_apply(dnsb_solver *s, MgLevel *L, const double *x,
                       double *y, double alpha, bool with_mass) {
  dnsb_ctx *ctx = s->ctx;
  const int n = L->n, nb = s->nb;
  const double *ad = with_mass ? s->mp_dinv.p : nullptr;
  const double *as = with_mass ? s->mp_scale.p : nullptr;
  if (L->tc.ok) {
    const TcPlan &p = L->tc;
    int tmem_cols = 32;
    while (tmem_cols < p.np_) tmem_cols *= 2;
    LAUNCH(ctx, k_tc_pack_x, dim3(cdiv(p.ldx, 32), cdiv(nb, 32)), 256, 0, x, L->xt.p, n, nb, p.ldx);
    LAUNCH(ctx, k_schur_tc, dim3(p.mtiles, p.splits), TC_THREADS, p.smem, (const float *)L->dinv_f32.p, p.mapB, L->tcpart.p, p.np_,
           p.kblocks, p.kb_per_split, p.stages, tmem_cols, g_schur_l2keep);
    LAUNCH(ctx, k_tc_epilogue, cdiv((size_t)n * nb, 256), 256, 0, (const float *)L->tcpart.p, p.splits,
           (size_t)p.mtiles * TC_BM * p.np_, p.np_, x, y, n, nb, alpha, ad, as);
    return 0;
  }
  if (nb <= 8)
    LAUNCH_N4(ctx, k_dense_gemv, nb <= 1, 1, nb <= 2, 2, nb <= 4, 4, 8, cdiv((size_t)n * 32, 256), 256, 0,
              L->dinv_dense.p, x, y, n, nb, alpha, ad, as);
  else {
    int tn;
    DenseSplit sp;
    dense_split(ctx, n, nb, &tn, &sp);
    const dim3 grid(sp.nctas, cdiv(nb, tn));
    if (g_schur_tf32 && L->dinv_f32.p && L->x_f32.p && tn == 64) {
      LAUNCH(ctx, k_f64_to_f32, cdiv((size_t)n * nb, 256), 256, 0, x, L->x_f32.p, (size_t)n, (size_t)nb, (size_t)nb);
      LAUNCH_N3(ctx, k_dense_tf32_streamk, g_schur_tf32 == 1, 3, g_schur_tf32 == 2, 2, 1, grid, 128, TFM_SMEM_BYTES,
                (const float *)L->dinv_f32.p, L->ldf, (const float *)L->x_f32.p, L->gpart.p, n, nb, sp);
    } else if (g_dmma && nb > 32 && n % 2 == 0 && nb % 2 == 0)
      LAUNCH(ctx, k_dense_dmma_streamk, grid, 128, DMM_SMEM_BYTES, L->dinv_dense.p, x, L->gpart.p, n, nb, sp);
    else
      LAUNCH_N3(ctx, k_dense_gemm_streamk, tn == 16, 16, tn == 32, 32, 64, grid, 128, 0, L->dinv_dense.p, x,
                L->gpart.p, n, nb, sp);
    LAUNCH(ctx, k_dense_epilogue, cdiv((size_t)n * nb, 256), 256, 0, (const double *)L->gpart.p, sp, x,
           y, n, nb, alpha, ad, as);
  }
  return 0;
}

// z = (k-step Jacobi-Chebyshev)(A) (r - C*zc)  with zero initial guess.
// C/zc: optional coupling (the gradient block of the preconditioner); `res`
// may alias r when there is no coupling.
static void cheb_run(dnsb_solver *s, const dnsb_csr *A, const double *coef,
                     const double *dinv, const dnsb_csr *C, const double *zc,
                     const double *r, double *z, double *res, double *d0, double *d1,
                     int k, double lmin, double lmax) {
  dnsb_ctx *ctx = s->ctx;
  const int nb = s->nb, n = A->nrows;
  const size_t nn = (size_t)n * nb;
  const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin);
  const double sigma = theta / delta;
  double rho = 1.0 / sigma;
  const bool batched = batched_ok(A, nb) && (!C || batched_ok(C, nb));
  const bool has2 = A->has2 && coef;
  double *dfirst = k == 1 ? z : d0;
  const int gpc = batched ? spb_gpc(ctx, n, nb) : 1;
  const bool pair = pair_ok(A, nb) && (!C || pair_ok(C, nb));
  // all rows pair up (both components of every node are unknowns)?
  const bool rowpair = pair && rowpairs_of(A, nb) * 2 == n;
  // fp32 smoother (dnsb_tile.cuh): fp64 in (r, zc), fp64 out (z), work vectors and matrix values fp32
  const bool f32 = g_cheb_f32 && C && A == s->F && s->cf_res.p && rowpair && has2 && nb == TILE_NB && A->tile.ok &&
                   k >= 2 && rowpairs_of(C, nb) * 2 == n;
  if (f32) {
    if (g_init_tile && C->tile.ok && C->tile.npairs == n / 2) {
      const TilePlan &cp = C->tile;
      const int per_sm_i = 2 * (cp.smem + 2048) <= (size_t)227 * 1024 ? 2 : 1;
      LAUNCH(ctx, k_cheb_init_tilef, std::min(cp.ntiles, per_sm_i * ctx->sm_count), TILE_THREADS, cp.smem, C->tile_view(), zc,
             D2C(r), (const float2 *)s->cf_dinv.p, (float2 *)s->cf_res.p, (float2 *)s->cf_d0.p, (float)(1.0 / theta));
    } else {
      LAUNCH(ctx, k_cheb_init_p2f, spp_grid(n / 2, nb), SPB_THREADS, 0, C->view(), D2C(zc), D2C(r),
             (const float2 *)s->cf_dinv.p, (float2 *)s->cf_res.p, (float2 *)s->cf_d0.p, nb, n / 2, (float)(1.0 / theta));
    }
  } else if (C) {
    if (pair && rowpairs_of(C, nb) * 2 == n)
      LAUNCH(ctx, k_cheb_init_p2, spp_grid(n / 2, nb), SPB_THREADS, 0, C->view(), D2C(zc), D2C(r),
             D2C(dinv), D2(res), D2(dfirst), nb, n / 2, 1.0 / theta);
    else if (pair)
      LAUNCH(ctx, k_cheb_init_b2, spb2_grid(n, nb), SPB_THREADS, 0, C->view(), D2C(zc), D2C(r),
             D2C(dinv), D2(res), D2(dfirst), nb, 1.0 / theta);
    else if (batched)
      LAUNCH(ctx, k_cheb_init_b, spb_grid(n, nb, gpc), SPB_THREADS, 0, C->view(), zc, r, dinv, res,
             dfirst, nb, gpc, 1.0 / theta);
    else if (spt_ok(C, nb)) {
      SptEpi ep{r, dinv, res, dfirst, nullptr, 1.0 / theta, 0.0};
      spt_launch_epi<SPT_CHEB_INIT>(ctx, C, nullptr, zc, ep);
    } else if (nb == 1)
      LAUNCH(ctx, k_cheb_init<8>, cdiv((size_t)n * 8, 256), 256, 0, C->view(), zc, r, dinv, res,
             dfirst, nb, 1.0 / theta);
    else
      LAUNCH(ctx, k_cheb_init<1>, cdiv(nn, 256), 256, 0, C->view(), zc, r, dinv, res, dfirst, nb,
             1.0 / theta);
  } else {
    LAUNCH(ctx, k_cheb_init_plain, cdiv(nn, 256), 256, 0, r, dinv, res, dfirst, nn, 1.0 / theta);
  }
  double *dc = d0, *dn = d1;
  float *dcf = s->cf_d0.p, *dnf = s->cf_d1.p;
  for (int i = 0; i + 1 < k; ++i) {
    const double rho_n = 1.0 / (2.0 * sigma - rho);
    const double c1 = rho_n * rho, c2 = 2.0 * rho_n / delta;
    const bool first = i == 0, last = i + 2 == k;
    if (f32) {
      const int per_sm = (g_tilef_ctas >= 2 && 2 * (A->tile.smem_f + 2048) <= (size_t)227 * 1024) ? 2 : 1;
      LAUNCH_BB(ctx, k_cheb_step_tilef, first, last, std::min(A->tile.ntiles, per_sm * ctx->sm_count), TILE_THREADS,
                A->tile.smem_f, A->tile_view_f(), coef, (const float *)dcf, (const float *)s->cf_dinv.p, s->cf_res.p,
                dnf, s->cf_z.p, z, (float)c1, (float)c2);
    } else if (rowpair && has2 && nb == TILE_NB && A->tile.ok) {
      // everything staged by TMA (dnsb_tile.cuh): persistent CTAs, one per SM
      LAUNCH_BB(ctx, k_cheb_step_tile, first, last, std::min(A->tile.ntiles, ctx->sm_count), TILE_THREADS,
                A->tile.smem, A->tile_view(), coef, (const double *)dc, dinv, res, dn, z, c1, c2);
    } else if (rowpair) {
      LAUNCH_BBB(ctx, k_cheb_step_p2, has2, first, last, spp_grid(n / 2, nb), SPB_THREADS, 0, A->view(), coef,
                 D2C(dc), D2C(dinv), D2(res), D2(dn), D2(z), nb, n / 2, c1, c2);
    } else if (pair) {
      LAUNCH_BBB(ctx, k_cheb_step_b2, has2, first, last, spb2_grid(n, nb), SPB_THREADS, 0, A->view(), coef,
                 D2C(dc), D2C(dinv), D2(res), D2(dn), D2(z), nb, c1, c2);
    } else if (batched) {
      LAUNCH_BBB(ctx, k_cheb_step_b, has2, first, last, spb_grid(n, nb, gpc), SPB_THREADS, 0, A->view(), coef,
                 (const double *)dc, dinv, res, dn, z, nb, gpc, c1, c2);
    } else if (spt_ok(A, nb)) {
      static constexpr decltype(&spt_launch_epi<SPT_CHEB_STEP>) step[2][2] = {
          {spt_launch_epi<SPT_CHEB_STEP>, spt_launch_epi<SPT_CHEB_STEP_LAST>},
          {spt_launch_epi<SPT_CHEB_STEP_FIRST>, spt_launch_epi<SPT_CHEB_STEP_ONLY>}};   // [first][last]
      step[first][last](ctx, A, coef, dc, SptEpi{nullptr, dinv, res, dn, z, c1, c2});
    } else if (nb == 1) {
      LAUNCH_XBB(ctx, k_cheb_step, 8, first, last, cdiv((size_t)n * 8, 256), 256, 0, A->view(), coef,
                 (const double *)dc, dinv, res, dn, z, nb, c1, c2);
    } else {
      LAUNCH_XBB(ctx, k_cheb_step, 1, first, last, cdiv(nn, 256), 256, 0, A->view(), coef, (const double *)dc, dinv,
                 res, dn, z, nb, c1, c2);
    }
    std::swap(dc, dn);
    std::swap(dcf, dnf);
    rho = rho_n;
  }
}

// out[i,m] = alpha*(a[i,m] + b[i,m]*rowscale[i])
__global__ void k_rowscale_add(const double *a, const double *b, const double *rowscale,
                               double *out, int n, int nb, double alpha) {
  dnsb_pdl_entry();
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)n * nb) return;
  out[t] = alpha * (a[t] + b[t] * rowscale[t / nb]);
}

// out[i,m] = alpha*a[i,m]*rowscale[i]
__global__ void k_rowscale_mul(const double *a, const double *rowscale, double *out, int n,
                               int nb, double alpha) {
  dnsb_pdl_entry();
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)n * nb) return;
  out[t] = alpha * a[t] * rowscale[t / nb];
}

// x = Vcycle(b) on level l of hierarchy `lv` (b, x: n_l*nb device vectors,
// b is not modified)
static void mg_vcycle(dnsb_solver *s, const std::vector<std::unique_ptr<MgLevel>> &lv, size_t l,
                      const double *b, double *x) {
  dnsb_ctx *ctx = s->ctx;
  MgLevel *L = lv[l].get();
  const int nb = s->nb;
  if (L->kind == MG_DENSE) {
    dense_apply(s, L, b, x, 1.0, false);
    return;
  }
  if (L->kind == MG_SMOOTH) {
    cheb_run(s, L->A, L->coef, L->dinv, nullptr, nullptr, b, x, L->r.p, L->d0.p, L->d1.p, L->nsmooth, L->lmin, L->lmax);
    return;
  }
  const size_t nn = (size_t)L->n * nb;
  MgLevel *C = lv[l + 1].get();
  // pre-smoothing from a zero guess
  cheb_run(s, L->A, L->coef, L->dinv, nullptr, nullptr, b, x, L->r.p, L->d0.p, L->d1.p, L->nsmooth, L->lmin, L->lmax);
  // residual and restriction
  spmm_dev(ctx, L->A, L->coef, x, b, L->r.p, nb, -1.0, 1.0);
  spmm_dev(ctx, L->R, nullptr, L->r.p, nullptr, C->b.p, nb, 1.0, 0.0);
  mg_vcycle(s, lv, l + 1, C->b.p, C->x.p);
  // prolongation and correction
  spmm_dev(ctx, L->P, nullptr, C->x.p, x, x, nb, 1.0, 1.0);
  // post-smoothing:  x += cheb(b - A x)
  spmm_dev(ctx, L->A, L->coef, x, b, L->r.p, nb, -1.0, 1.0);
  cheb_run(s, L->A, L->coef, L->dinv, nullptr, nullptr, L->r.p, L->t.p, L->r.p, L->d0.p, L->d1.p,
           L->nsmooth, L->lmin, L->lmax);
  LAUNCH(ctx, k_axpby, cdiv(nn, 256), 256, 0, 1.0, (const double *)x, 1.0, (const double *)L->t.p, x, nn);
}

// x = alpha * L^-1 b  with the pressure hierarchy (dense inverse or V-cycle)
static void schur_levels_apply(dnsb_solver *s, const double *b, double *x, double alpha) {
  dnsb_ctx *ctx = s->ctx;
  const size_t npb = (size_t)s->np * s->nb;
  MgLevel *L0 = s->levels[0].get();
  if (L0->kind == MG_DENSE) {
    dense_apply(s, L0, b, x, alpha, false);
  } else {
    mg_vcycle(s, s->levels, 0, b, L0->x.p);
    LAUNCH(ctx, k_axpby, cdiv(npb, 256), 256, 0, alpha, (const double *)L0->x.p, 0.0,
           (const double *)nullptr, x, npb);
  }
}

// z = P^-1 r   (block upper-triangular preconditioner)
static int apply_prec(dnsb_solver *s, const double *r, double *z) {
  dnsb_ctx *ctx = s->ctx;
  const int nb = s->nb, nv = s->nv, np = s->np;
  const size_t nvb = (size_t)nv * nb, npb = (size_t)np * nb;
  const double *rv = r, *rp = r + nvb;
  double *zv = z, *zp = z + nvb;
  DNSB_REQUIRE(ctx, !s->levels.empty() || s->has_mass, "no Schur approximation set");
  if (s->prec_diag) {
    // diag(Fh^-1, +Sh^-1): no gradient coupling, positive Schur block -- the symmetric positive definite
    // preconditioner MINRES needs (Chebyshev polynomial of the symmetric F, dense inverse of J Z JT)
    DNSB_REQUIRE(ctx, !s->has_lsc && !s->levels.empty() && s->levels[0]->kind == MG_DENSE &&
                          s->vlevels[0]->kind == MG_SMOOTH,
                 "block-diagonal preconditioner: Chebyshev velocity block + dense Schur block only");
    DNSB_CK(ctx, s->zero_p.alloc(npb));
    DNSB_CK(ctx, s->zero_p.zero(ctx->stream));
    dense_apply(s, s->levels[0].get(), rp, zp, 1.0, s->has_mass);
    cheb_run(s, s->F, s->has_coef ? s->coef.p : nullptr, s->dinv.p, s->JT, s->zero_p.p, rv, zv, s->cres.p,
             s->cd0.p, s->cd1.p, s->kF, s->lmin, s->lmax);
    return 0;
  }
  // ---- zp = -Sh^-1 rp ------------------------------------------------------
  if (s->has_lsc) {
    // least-squares commutator (Elman et al. 2006):
    //   Sh^-1 = L^-1 (J Du^-1 F Du^-1 JT) L^-1,   L = J Du^-1 JT
    const double *coef = s->has_coef ? s->coef.p : nullptr;
    schur_levels_apply(s, rp, s->lsc_p1.p, 1.0);
    spmm_dev(ctx, s->JT, nullptr, s->lsc_p1.p, nullptr, s->lsc_t1.p, nb, 1.0, 0.0);
    LAUNCH(ctx, k_rowscale_mul, cdiv(nvb, 256), 256, 0, s->lsc_t1.p, s->lsc_dinv.p, s->lsc_t1.p, nv, nb, 1.0);
    spmm_dev(ctx, s->F, coef, s->lsc_t1.p, nullptr, s->lsc_t2.p, nb, 1.0, 0.0);
    LAUNCH(ctx, k_rowscale_mul, cdiv(nvb, 256), 256, 0, s->lsc_t2.p, s->lsc_dinv.p, s->lsc_t2.p, nv, nb, 1.0);
    spmm_dev(ctx, s->J, nullptr, s->lsc_t2.p, nullptr, s->lsc_p2.p, nb, 1.0, 0.0);
    schur_levels_apply(s, s->lsc_p2.p, zp, -1.0);
  } else if (s->levels.empty()) {
    // scaled (lumped) pressure mass matrix only:  zp = -scale_m * mp_dinv_i * rp
    LAUNCH(ctx, k_scale_member, cdiv(npb, 256), 256, 0, rp, s->mp_scale.p, zp, (size_t)np, nb);
    LAUNCH(ctx, k_rowscale_mul, cdiv(npb, 256), 256, 0, zp, s->mp_dinv.p, zp, np, nb, -1.0);
  } else {
    MgLevel *L0 = s->levels[0].get();
    if (L0->kind == MG_DENSE) {
      dense_apply(s, L0, rp, zp, -1.0, s->has_mass);
    } else {
      mg_vcycle(s, s->levels, 0, rp, L0->x.p);
      if (s->has_mass) {
        // t = scale_m*rp ;  zp = -(x + mp_dinv_i*t)
        LAUNCH(ctx, k_scale_member, cdiv(npb, 256), 256, 0, rp, s->mp_scale.p, L0->t.p, (size_t)np, nb);
        LAUNCH(ctx, k_rowscale_add, cdiv(npb, 256), 256, 0, L0->x.p, L0->t.p, s->mp_dinv.p, zp, np, nb, -1.0);
      } else {
        LAUNCH(ctx, k_axpby, cdiv(npb, 256), 256, 0, -1.0, (const double *)L0->x.p, 0.0,
               (const double *)nullptr, zp, npb);
      }
    }
  }
  // ---- zv = Fh^-1 (rv - JT zp) ---------------------------------------------
  MgLevel *V0 = s->vlevels[0].get();
  if (V0->kind != MG_SMOOTH) {
    spmm_dev(ctx, s->JT, nullptr, zp, rv, V0->b.p, nb, -1.0, 1.0);
    mg_vcycle(s, s->vlevels, 0, V0->b.p, zv);
    return 0;
  }
  // single level: Chebyshev only, fused with the gradient coupling
  cheb_run(s, s->F, s->has_coef ? s->coef.p : nullptr, s->dinv.p, s->JT, zp, rv, zv, s->cres.p,
           s->cd0.p, s->cd1.p, s->kF, s->lmin, s->lmax);
  return 0;
}

// One Arnoldi step of FGMRES (column j): z_j = P^-1 v_j, w = K z_j, Gram-Schmidt
// against v_0..v_j, Givens update, v_{j+1}.  All arguments are fixed device
// buffers, so the launch sequence of a column is captured once as a CUDA graph
// and replayed (one graph launch instead of ~20 kernel launches: the single
// trajectory is launch-latency bound, SURVEY.md 8d).
static int gmres_iteration_launch(dnsb_solver *s, int j, double tol) {
  dnsb_ctx *ctx = s->ctx;
  const int nb = s->nb, ntot = s->ntot;
  const size_t ntb = (size_t)ntot * nb;
  const RedCfg &rc = s->rc;
  const double *coef = s->has_coef ? s->coef.p : nullptr;
  double *Vj = s->Vb.p + (size_t)j * ntb;
  double *Zj = s->Zb.p + (size_t)j * ntb;
  if (apply_prec(s, Vj, Zj)) return -1;
  spmm_dev(ctx, s->K.get(), coef, Zj, nullptr, s->w.p, nb, 1.0, 0.0);
  // classical Gram-Schmidt; a second pass (CGS2) for long recurrences,
  // where one pass loses the orthogonality of the basis and FGMRES stalls
  // (the Oseen/Newton systems of the steady solver need 150-300 iterations)
  const bool reorth = (nb == 1) || j >= 16;
  double *Vn = s->Vb.p + (size_t)(j + 1) * ntb;
  mdot_dev(ctx, rc, s->Vb.p, ntb, j + 1, s->w.p, ntot, nb, s->partial.p, s->gs.h);
  if (!reorth && s->use_pyth) {
    // one pass less and no scalar glue: the norm of the orthogonalised vector from Pythagoras,
    // Givens first, then the update writes the NORMALISED vector (no k_scale_member pass, no
    // reduction of 586 partial norms inside the one-CTA Givens kernel)
    {
      const size_t gsm = (size_t)3 * (j + 2) * nb * sizeof(double);
      const int staged = gsm <= 96 * 1024;
      LAUNCH(ctx, k_gmres_givens, 1, 1024, staged ? gsm : 0, s->gs, (const double *)nullptr, 0, nb, j, tol, 1, staged);
    }
    gs_update_dev(ctx, rc, s->Vb.p, ntb, j + 1, s->gs.h, s->w.p, Vn, ntot, nb, s->partial2.p,
                  (const double *)s->gs.invh);
    return 0;
  }
  gs_update_dev(ctx, rc, s->Vb.p, ntb, j + 1, s->gs.h, s->w.p, Vn, ntot, nb, s->partial2.p);
  const double *unscaled = Vn;
  if (reorth) {
    mdot_dev(ctx, rc, s->Vb.p, ntb, j + 1, Vn, ntot, nb, s->partial.p, s->gh2.p);
    gs_update_dev(ctx, rc, s->Vb.p, ntb, j + 1, s->gh2.p, Vn, s->w.p, ntot, nb, s->partial2.p);
    LAUNCH(ctx, k_axpby, cdiv((size_t)(j + 1) * nb, 256), 256, 0, 1.0, (const double *)s->gs.h, 1.0,
           (const double *)s->gh2.p, s->gs.h, (size_t)(j + 1) * nb);
    unscaled = s->w.p;
  }
  {
    const size_t gsm = (size_t)3 * (j + 2) * nb * sizeof(double);
    const int staged = gsm <= 96 * 1024;
    LAUNCH(ctx, k_gmres_givens, 1, 1024, staged ? gsm : 0, s->gs, (const double *)s->partial2.p, rc.nblocks, nb, j, tol, 0, staged);
  }
  LAUNCH(ctx, k_scale_member, cdiv(ntb, 256), 256, 0, unscaled, (const double *)s->gs.invh, Vn,
         (size_t)ntot, nb);
  return 0;
}

static void solver_drop_graphs(dnsb_solver *s) {
  if (s->igraph.empty() && s->mr <= 0) return;
  for (cudaGraphExec_t g : s->igraph) if (g) cudaGraphExecDestroy(g);
  s->igraph.assign(s->mr, nullptr);
  s->igraph_launches.assign(s->mr, 0);
  s->igraph_seen.assign(s->mr, 0);
}

static int gmres_iteration(dnsb_solver *s, int j, double tol) {
  dnsb_ctx *ctx = s->ctx;
  if (!g_graphs || ctx->prof) return gmres_iteration_launch(s, j, tol);
  if (s->igraph.empty() || s->igraph_tol != tol || s->igraph_pyth != s->use_pyth) {
    solver_drop_graphs(s);
    s->igraph_tol = tol;
    s->igraph_pyth = s->use_pyth;
  }
  // a column is captured the SECOND time it runs: capture + instantiation cost more than the launches of one
  // pass, so one-shot solvers (a steady Picard/Newton system, 200 columns used once) stay on plain launches
  if (!s->igraph[j] && s->igraph_seen[j]++ == 0) return gmres_iteration_launch(s, j, tol);
  if (!s->igraph[j]) {
    const long long l0 = ctx->launches;
    cudaGraph_t graph = nullptr;
    DNSB_CK(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    const int rc = gmres_iteration_launch(s, j, tol);
    const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
    if (rc || e != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      if (!rc) DNSB_CK(ctx, e);
      return -1;
    }
    s->igraph_launches[j] = (int)(ctx->launches - l0);
    ctx->launches = l0;
    cudaGraphExec_t ex = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&ex, graph, 0);
    cudaGraphDestroy(graph);
    DNSB_CK(ctx, e2);
    s->igraph[j] = ex;
  }
  DNSB_CK(ctx, cudaGraphLaunch(s->igraph[j], ctx->stream));
  ctx->launches += s->igraph_launches[j];
  return 0;
}

static int read_flags(dnsb_solver *s) {
  dnsb_ctx *ctx = s->ctx;
  DNSB_CK(ctx, cudaMemcpyAsync(s->h_flags.p, s->gs.flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

// FGMRES on device vectors: b (ntot*nb), x (in: initial guess, out: solution)
static int solver_solve_dev(dnsb_solver *s, const double *b, double *x, double tol,
                            int maxit, bool zero_guess) {
  dnsb_ctx *ctx = s->ctx;
  const int nb = s->nb, ntot = s->ntot, mr = s->mr;
  const size_t ntb = (size_t)ntot * nb;
  const RedCfg &rc = s->rc;
  const double *coef = s->has_coef ? s->coef.p : nullptr;
  // |b|
  LAUNCH(ctx, k_dot1, rc.nblocks, rc.threads, rc.smem, b, b, ntot, nb, rc.rpb, s->partial2.p);
  LAUNCH(ctx, k_reduce_partials2, cdiv(nb, 32), 1024, 0, (const double *)s->partial2.p, rc.nblocks, nb, s->red.p);
  LAUNCH(ctx, k_set_bnorm, 1, std::max(32, ((nb + 31) / 32) * 32), 0, s->gs, (const double *)s->red.p, 1, nb);
  if (zero_guess) DNSB_CK(ctx, cudaMemsetAsync(x, 0, ntb * sizeof(double), ctx->stream));
  int total = 0;
  bool first = true;
  int expect = s->expect_its;
  s->use_pyth = g_gs_pyth && nb > 1 && expect >= 1 && expect <= 8;
  while (true) {
    double *V0 = s->Vb.p;
    if (zero_guess && first)
      DNSB_CK(ctx, cudaMemcpyAsync(V0, b, ntb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    else
      spmm_dev(ctx, s->K.get(), coef, x, b, V0, nb, -1.0, 1.0);
    LAUNCH(ctx, k_dot1, rc.nblocks, rc.threads, rc.smem, V0, V0, ntot, nb, rc.rpb, s->partial2.p);
    LAUNCH(ctx, k_reduce_partials2, cdiv(nb, 32), 1024, 0, (const double *)s->partial2.p, rc.nblocks, nb, s->red.p);
    LAUNCH(ctx, k_gmres_begin, 1, std::max(32, ((nb + 31) / 32) * 32), 0, s->gs, (const double *)s->red.p,
           1, nb, tol, first ? 1 : 0);
    LAUNCH(ctx, k_scale_member, cdiv(ntb, 256), 256, 0, V0, s->gs.invh, V0, (size_t)ntot, nb);
    first = false;
    if (read_flags(s)) return -1;
    if (s->h_flags.p[0] == 0) break;
    int j = 0;
    bool alldone = false;
    for (; j < mr && total < maxit; ++j, ++total) {
      if (gmres_iteration(s, j, tol)) return -1;
      // convergence poll: skipped while far from the expected iteration count
      if (total + 1 >= expect - 1 || j + 1 == mr || total + 1 == maxit) {
        if (read_flags(s)) return -1;
        if (s->h_flags.p[0] == 0) { alldone = true; ++j; ++total; break; }
      }
    }
    const int ncols = j;
    if (ncols > 0) {
      LAUNCH(ctx, k_gmres_solve_y, 1, std::max(32, ((nb + 31) / 32) * 32), 0, s->gs, nb, ncols);
      LAUNCH(ctx, k_gmres_update_x, cdiv(ntb, 256), 256, 0, s->Zb.p, ntb, ncols, s->gs.h, x,
             (size_t)ntot, nb);
    }
    if (alldone || total >= maxit) break;
  }
  if (s->h_flags.p[0] != 0) {
    // stopped at maxit: the residual of the unfinished members enters the
    // running maximum, the solve is counted (callers decide what to do)
    LAUNCH(ctx, k_gmres_track_unconverged, 1, std::max(32, ((nb + 31) / 32) * 32), 0, s->gs, nb);
    s->stat_unconverged += 1;
  }
  // h_flags[1]: iteration at which the last member converged (<= total; the
  // difference are iterations launched between two convergence polls)
  const int needed = std::min(total, std::max(0, s->h_flags.p[1]));
  s->expect_its = needed;
  s->stat_iters += needed;
  s->stat_launched += total;
  s->stat_solves += 1;
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// max over members of the running maximum of the final relative residuals
// since the last reset (NaN if any solve produced one); optionally reset
static int solver_relmax_members(dnsb_solver *s, std::vector<double> &h, bool reset = false) {
  dnsb_ctx *ctx = s->ctx;
  h.resize(s->nb);
  DNSB_CK(ctx, cudaMemcpyAsync(h.data(), s->grelmax.p, s->nb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (reset) DNSB_CK(ctx, s->grelmax.zero(ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}
static int solver_relmax(dnsb_solver *s, bool reset, double *out) {
  std::vector<double> h;
  if (solver_relmax_members(s, h, reset)) return -1;
  double mx = 0.0;
  for (int m = 0; m < s->nb; ++m) {
    if (h[m] != h[m]) { mx = h[m]; break; }   // NaN wins
    if (h[m] > mx) mx = h[m];
  }
  *out = mx;
  return 0;
}

extern "C" int dnsb_solver_solve(dnsb_solver *s, const double *rhsv, const double *rhsp,
                                 const double *x0, double *vp, double tol, int maxit,
                                 int *iters, double *relres) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, rhsv && vp && maxit >= 1 && tol > 0, "bad arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int nb = s->nb;
  const size_t nvb = (size_t)s->nv * nb, npb = (size_t)s->np * nb, ntb = nvb + npb;
  DNSB_CK(ctx, s->sb.alloc(ntb));
  DNSB_CK(ctx, s->sx.alloc(ntb));
  DNSB_CK(ctx, cudaMemcpyAsync(s->sb.p, rhsv, nvb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (rhsp)
    DNSB_CK(ctx, cudaMemcpyAsync(s->sb.p + nvb, rhsp, npb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  else
    DNSB_CK(ctx, cudaMemsetAsync(s->sb.p + nvb, 0, npb * sizeof(double), ctx->stream));
  if (x0)
    DNSB_CK(ctx, cudaMemcpyAsync(s->sx.p, x0, ntb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  s->expect_its = 0;
  int rc = solver_solve_dev(s, s->sb.p, s->sx.p, tol, maxit, x0 == nullptr);
  if (rc) return rc;
  DNSB_CK(ctx, cudaMemcpyAsync(vp, s->sx.p, ntb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<double> res(nb), bn(nb);
  std::vector<int> it(nb);
  DNSB_CK(ctx, cudaMemcpyAsync(res.data(), s->gs.resid, nb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaMemcpyAsync(bn.data(), s->gs.bnorm, nb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaMemcpyAsync(it.data(), s->gs.ittot, nb * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  for (int m = 0; m < nb; ++m) {
    if (iters) iters[m] = it[m];
    if (relres) relres[m] = bn[m] > 0 ? res[m] / bn[m] : 0.0;
  }
  return 0;
}

// K.v1[kpos(i, k)] = F.v1[k] for the entries k of row i of F (K row i holds the
// F entries first, then the JT entries)
__global__ void k_copy_f_into_k(CsrDev F, const int *__restrict__ kindptr,
                                double *__restrict__ kv1) {
  dnsb_pdl_entry();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= F.nrows) return;
  const int f0 = F.indptr[row], f1 = F.indptr[row + 1], k0 = kindptr[row];
  for (int k = f0 + lane; k < f1; k += 32) kv1[k0 + (k - f0)] = F.v1[k];
}

// New values of the velocity block on the unchanged pattern (Picard/Newton
// and Crank-Nicolson sweeps: stokes_navier_utils.py:1484-1512 builds and
// factorises a new matrix every step; here only the values move, the
// preconditioner set-up -- Schur approximation, Chebyshev bounds -- is kept).
extern "C" int dnsb_solver_update_fvalues(dnsb_solver *s, const double *vals1) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, vals1 != nullptr, "null values");
  DNSB_REQUIRE(ctx, !s->F->has2, "matrices with two value arrays are updated through their coefficients");
  DNSB_CK(ctx, dnsb_enter(ctx));
  dnsb_csr *F = s->F;
  DNSB_CK(ctx, cudaMemcpyAsync(F->v1.p, vals1, (size_t)F->nnz * sizeof(double), cudaMemcpyHostToDevice,
                               ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));   // host buffer is borrowed
  std::copy(vals1, vals1 + F->nnz, F->h_v1.begin());
  F->tile.ok = false;   // packed copies of the values are stale: the row-pair kernels serve this matrix
  s->K->tile.ok = false;
  LAUNCH(ctx, k_copy_f_into_k, cdiv((size_t)F->nrows * 32, 256), 256, 0, F->view(),
         (const int *)s->K->indptr.p, s->K->v1.p);
  const size_t nvb = (size_t)s->nv * s->nb;
  LAUNCH(ctx, k_diag_inv, cdiv(nvb, 256), 256, 0, F->view(), s->diagpos.p,
         (const double *)nullptr, s->dinv.p, s->nb);
  s->expect_its = 0;
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// ===========================================================================
// device-resident Picard/Newton + Crank-Nicolson sweep
// ===========================================================================
// vals[pos[k]] = n1[src[k]] (+ n2[src[k]]);  vals is zeroed by the caller
__global__ void k_conv_to_pattern(const double *__restrict__ n1, const double *__restrict__ n2,
                                  const int *__restrict__ src, const int *__restrict__ pos,
                                  double *__restrict__ vals, int nconv) {
  dnsb_pdl_entry();
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nconv) return;
  const int sk = src[k];
  vals[pos[k]] = n2 ? n1[sk] + n2[sk] : n1[sk];
}

// out[i] = fv[i] - sum_k (n1[k] (+ n2[k])) * ubc[col_k]  over row inv[i] of the
// full convection pattern  (+ f3[inv[i]] for Newton);  8 lanes per row
__global__ void k_conv_rhs(const int *__restrict__ cindptr, const int *__restrict__ cindices,
                           const double *__restrict__ n1, const double *__restrict__ n2,
                           const double *__restrict__ ubc, const double *__restrict__ f3,
                           const double *__restrict__ fv, const int *__restrict__ inv,
                           double *__restrict__ out, int nv) {
  dnsb_pdl_entry();
  const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int i = (int)(tid >> 3), lane = (int)(tid & 7);
  double acc = 0.0;
  if (i < nv) {
    const int r = inv[i];
    for (int k = cindptr[r] + lane; k < cindptr[r + 1]; k += 8)
      acc += (n2 ? n1[k] + n2[k] : n1[k]) * ubc[cindices[k]];
  }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, 8);
  if (i < nv && lane == 0) out[i] = fv[i] - acc + (f3 ? f3[inv[i]] : 0.0);
}

// out = a + c*(b + n)   (value arrays on one pattern)
__global__ void k_vals_combine(const double *__restrict__ a, const double *__restrict__ b,
                               const double *__restrict__ n, double c, double *__restrict__ out,
                               size_t nnz) {
  dnsb_pdl_entry();
  size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  out[k] = a[k] + c * (b[k] + n[k]);
}

// rhs = rhs + c*(fa + fb - y)
__global__ void k_cn_rhs(double *__restrict__ rhs, const double *__restrict__ fa,
                         const double *__restrict__ fb, const double *__restrict__ y, double c,
                         int n) {
  dnsb_pdl_entry();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rhs[i] += c * (fa[i] + fb[i] - y[i]);
}

// d = v - lin[inv]   (difference to the linearisation point, inner dofs)
__global__ void k_diff_inner(const double *__restrict__ v, const double *__restrict__ linfull,
                             const int *__restrict__ inv, double *__restrict__ d, int nv) {
  dnsb_pdl_entry();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  d[i] = v[i] - linfull[inv[i]];
}

struct dnsb_cnsweep {
  dnsb_ctx *ctx = nullptr;
  unsigned long long mesh_hash = 0;
  dnsb_solver *s = nullptr;
  dnsb_csr *M = nullptr;      // mass matrix (own pattern)
  std::unique_ptr<dnsb_csr> C;   // (A + N_c) on the pattern of F
  int nv = 0, np = 0, nvf = 0, nconv = 0, nbc = 0;
  DBuf<double> mv, av, nvn, nvc;          // value arrays on the pattern of F
  DBuf<int> src, pos, inv, bcinds;
  DBuf<double> bcvals, ubc, fv, fp;
  DBuf<double> n1, n2, f3;                // K1b outputs on the full convection pattern
  DBuf<double> vfull, fn, fc, b, x, xprev, xguess, y, dvec, mdv, lin, vtraj, ptraj, v, p;
  DBuf<double> npart, nout;
  double max_relres = 0;      // of the last sweep (all step solves)
  long long unconverged = 0;
  int guess_mode = 1;         // 0: previous solution ('old'), 1: linear extrapolation ('upd')
  ~dnsb_cnsweep() { cudaStreamSynchronize(ctx->stream); }   // no buffer is freed under a running kernel
};

extern "C" int dnsb_cnsweep_create(dnsb_solver *s, dnsb_csr *mmat, const double *mvals,
                                   const double *avals, int nconv, const int32_t *src,
                                   const int32_t *pos, const int32_t *invinds, int nbc,
                                   const int32_t *bcinds, const double *bcvals, const double *fv,
                                   const double *fp, dnsb_cnsweep **out) {
  if (out) *out = nullptr;
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, out && mmat && mvals && avals && src && pos && invinds && fv, "null arguments");
  DNSB_REQUIRE(ctx, s->nb == 1 && !s->F->has2, "the sweep needs a single-system solver with one value array");
  DNSB_REQUIRE(ctx, ctx->ncell > 0 && ctx->cnnz > 0, "set the mesh and the convection pattern first");
  DNSB_REQUIRE(ctx, mmat->nrows == s->nv && mmat->ncols == s->nv, "mass matrix shape");
  const int nv = s->nv, np = s->np, nvf = 2 * ctx->nnodes;
  const int nnz = s->F->nnz;
  for (int k = 0; k < nconv; ++k)
    DNSB_REQUIRE(ctx, src[k] >= 0 && src[k] < ctx->cnnz && pos[k] >= 0 && pos[k] < nnz, "convection map out of range");
  for (int i = 0; i < nv; ++i) DNSB_REQUIRE(ctx, invinds[i] >= 0 && invinds[i] < nvf, "invinds out of range");
  for (int i = 0; i < nbc; ++i) DNSB_REQUIRE(ctx, bcinds[i] >= 0 && bcinds[i] < nvf, "bcinds out of range");
  DNSB_CK(ctx, dnsb_enter(ctx));
  std::unique_ptr<dnsb_cnsweep> w(new (std::nothrow) dnsb_cnsweep());
  DNSB_REQUIRE(ctx, w != nullptr, "out of host memory");
  w->ctx = ctx; w->mesh_hash = ctx->mesh_hash; w->s = s; w->M = mmat;
  w->nv = nv; w->np = np; w->nvf = nvf; w->nconv = nconv; w->nbc = nbc;
  {
    int rc = csr_build(ctx, nv, nv, s->F->h_indptr.data(), s->F->h_indices.data(), avals, nullptr, w->C);
    if (rc) return rc;
  }
  DNSB_CK(ctx, w->mv.upload(mvals, nnz, ctx->stream));
  DNSB_CK(ctx, w->av.upload(avals, nnz, ctx->stream));
  DNSB_CK(ctx, w->nvn.alloc(nnz)); DNSB_CK(ctx, w->nvc.alloc(nnz));
  DNSB_CK(ctx, w->src.upload(src, nconv, ctx->stream));
  DNSB_CK(ctx, w->pos.upload(pos, nconv, ctx->stream));
  DNSB_CK(ctx, w->inv.upload(invinds, nv, ctx->stream));
  std::vector<double> ub(nvf, 0.0);
  for (int i = 0; i < nbc; ++i) ub[bcinds[i]] = bcvals[i];
  DNSB_CK(ctx, w->ubc.upload(ub.data(), nvf, ctx->stream));
  if (nbc > 0) {
    DNSB_CK(ctx, w->bcinds.upload(bcinds, nbc, ctx->stream));
    DNSB_CK(ctx, w->bcvals.upload(bcvals, nbc, ctx->stream));
  }
  std::vector<double> zero(np, 0.0);
  DNSB_CK(ctx, w->fv.upload(fv, nv, ctx->stream));
  DNSB_CK(ctx, w->fp.upload(fp ? fp : zero.data(), np, ctx->stream));
  DNSB_CK(ctx, w->n1.alloc(ctx->cnnz)); DNSB_CK(ctx, w->n2.alloc(ctx->cnnz));
  DNSB_CK(ctx, w->f3.alloc(nvf));
  DNSB_CK(ctx, w->vfull.alloc(nvf)); DNSB_CK(ctx, w->fn.alloc(nv)); DNSB_CK(ctx, w->fc.alloc(nv));
  DNSB_CK(ctx, w->b.alloc(nv + np)); DNSB_CK(ctx, w->x.alloc(nv + np)); DNSB_CK(ctx, w->y.alloc(nv));
  DNSB_CK(ctx, w->xprev.alloc(nv + np)); DNSB_CK(ctx, w->xguess.alloc(nv + np));
  DNSB_CK(ctx, w->dvec.alloc(nv)); DNSB_CK(ctx, w->mdv.alloc(nv));
  DNSB_CK(ctx, w->v.alloc(nv)); DNSB_CK(ctx, w->p.alloc(np));
  RedCfg rc = red_cfg(ctx, nv, 1);
  DNSB_CK(ctx, w->npart.alloc(rc.nblocks)); DNSB_CK(ctx, w->nout.alloc(1));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  *out = w.release();
  return 0;
}

extern "C" void dnsb_cnsweep_destroy(dnsb_cnsweep *w) {
  if (!w) return;
  dnsb_enter(w->ctx);
  delete w;
}

// values of the condensed convection matrix of `vfull` on the pattern of F
// (into `vals`) and f = fv - (N u_bc)[inv] (+ N(v)v[inv] for Newton)
static int cnsweep_conv(dnsb_cnsweep *w, const double *vfull, bool picard, double *vals, double *f) {
  dnsb_ctx *ctx = w->ctx;
  int rc = convmats_dev(ctx, vfull, w->n1.p, picard ? nullptr : w->n2.p, picard ? nullptr : w->f3.p);
  if (rc) return rc;
  const double *n2 = picard ? nullptr : w->n2.p;
  DNSB_CK(ctx, cudaMemsetAsync(vals, 0, (size_t)w->s->F->nnz * sizeof(double), ctx->stream));
  LAUNCH(ctx, k_conv_to_pattern, cdiv(w->nconv, 256), 256, 0, (const double *)w->n1.p, n2,
         (const int *)w->src.p, (const int *)w->pos.p, vals, w->nconv);
  LAUNCH(ctx, k_conv_rhs, cdiv((size_t)w->nv * 8, 256), 256, 0, (const int *)ctx->cindptr.p,
         (const int *)ctx->cindices.p, (const double *)w->n1.p, n2, (const double *)w->ubc.p,
         picard ? (const double *)nullptr : (const double *)w->f3.p, (const double *)w->fv.p,
         (const int *)w->inv.p, f, w->nv);
  return 0;
}

// One sweep over the time grid (stokes_navier_utils.py:1402-1566): step n
// linearises the "next" side about linpoint[n] (the previous sweep's state,
// full vectors incl. boundary values) and the "current" side about the
// sweep's own state.  dts: nsteps step sizes.  vtraj ((nsteps+1)*nvf) and
// ptraj ((nsteps+1)*np) receive the trajectory (index 0 = initial state);
// upd_norm = sum_n dt_n (v_n - lin_n)^T M (v_n - lin_n)  (:1557-1560).
extern "C" int dnsb_cnsweep_run(dnsb_cnsweep *w, int nsteps, const double *dts, int picard,
                                const double *linpoint, const double *v0, const double *p0,
                                double tol, int maxit, double *vtraj, double *ptraj,
                                double *upd_norm, long long *iters_total) {
  if (!w) return -2;
  dnsb_ctx *ctx = w->ctx;
  DNSB_REQUIRE(ctx, nsteps >= 1 && dts && linpoint && v0 && vtraj && ptraj, "bad arguments");
  DNSB_REQUIRE(ctx, w->mesh_hash == ctx->mesh_hash, "the mesh of the context is not the one this sweep was created on");
  DNSB_CK(ctx, dnsb_enter(ctx));
  dnsb_solver *s = w->s;
  const int nv = w->nv, np = w->np, nvf = w->nvf, nnz = s->F->nnz;
  DNSB_CK(ctx, w->lin.upload(linpoint, (size_t)(nsteps + 1) * nvf, ctx->stream));
  DNSB_CK(ctx, w->vtraj.alloc((size_t)(nsteps + 1) * nvf));
  DNSB_CK(ctx, w->ptraj.alloc((size_t)(nsteps + 1) * np));
  DNSB_CK(ctx, cudaMemcpyAsync(w->v.p, v0, nv * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (p0) DNSB_CK(ctx, cudaMemcpyAsync(w->p.p, p0, np * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  else DNSB_CK(ctx, w->p.zero(ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  RedCfg rcn = red_cfg(ctx, nv, 1);
  // full velocity of the initial state (boundary values included)
  DNSB_CK(ctx, w->vfull.zero(ctx->stream));
  if (w->nbc > 0)
    LAUNCH(ctx, k_set_bcs, cdiv((size_t)w->nbc, 256), 256, 0, w->bcinds.p, w->bcvals.p, w->vfull.p, w->nbc, 1);
  LAUNCH(ctx, k_scatter_inner, cdiv((size_t)nv, 256), 256, 0, (const double *)w->v.p, w->inv.p, w->vfull.p, nv, 1);
  DNSB_CK(ctx, cudaMemcpyAsync(w->vtraj.p, w->vfull.p, nvf * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  DNSB_CK(ctx, cudaMemcpyAsync(w->ptraj.p, w->p.p, np * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  int rc = cnsweep_conv(w, w->vfull.p, picard != 0, w->nvc.p, w->fc.p);
  if (rc) return rc;
  // x0 of the first solve: [v; -dt p]
  DNSB_CK(ctx, cudaMemcpyAsync(w->x.p, w->v.p, nv * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  LAUNCH(ctx, k_axpby, cdiv((size_t)np, 256), 256, 0, -dts[0], (const double *)w->p.p, 0.0,
         (const double *)nullptr, w->x.p + nv, (size_t)np);
  double norm_acc = 0.0;
  long long its0 = s->stat_iters;
  const long long unc0 = s->stat_unconverged;
  DNSB_CK(ctx, s->grelmax.zero(ctx->stream));
  for (int n = 1; n <= nsteps; ++n) {
    const double dt = dts[n - 1];
    const double *lin_n = w->lin.p + (size_t)n * nvf;
    // "next" side: linearised about the previous sweep's state at t_n
    rc = cnsweep_conv(w, lin_n, picard != 0, w->nvn.p, w->fn.p);
    if (rc) return rc;
    // F = M + dt/2 (A + N_n)  -> solver (values of F, its copy inside K, Jacobi diagonal)
    LAUNCH(ctx, k_vals_combine, cdiv((size_t)nnz, 256), 256, 0, (const double *)w->mv.p,
           (const double *)w->av.p, (const double *)w->nvn.p, 0.5 * dt, s->F->v1.p, (size_t)nnz);
    LAUNCH(ctx, k_copy_f_into_k, cdiv((size_t)nv * 32, 256), 256, 0, s->F->view(),
           (const int *)s->K->indptr.p, s->K->v1.p);
    LAUNCH(ctx, k_diag_inv, cdiv((size_t)nv, 256), 256, 0, s->F->view(), s->diagpos.p,
           (const double *)nullptr, s->dinv.p, 1);
    // rhs = M v + dt/2 (f_n + f_c - (A + N_c) v)
    LAUNCH(ctx, k_axpby, cdiv((size_t)nnz, 256), 256, 0, 1.0, (const double *)w->av.p, 1.0,
           (const double *)w->nvc.p, w->C->v1.p, (size_t)nnz);
    spmm_dev(ctx, w->C.get(), nullptr, w->v.p, nullptr, w->y.p, 1, 1.0, 0.0);
    spmm_dev(ctx, w->M, nullptr, w->v.p, nullptr, w->b.p, 1, 1.0, 0.0);
    LAUNCH(ctx, k_cn_rhs, cdiv(nv, 256), 256, 0, w->b.p, (const double *)w->fn.p, (const double *)w->fc.p,
           (const double *)w->y.p, 0.5 * dt, nv);
    DNSB_CK(ctx, cudaMemcpyAsync(w->b.p + nv, w->fp.p, np * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    // initial guess: linear extrapolation 2 x_{n-1} - x_{n-2} of the saddle
    // solutions (the reference's `krylovini='upd'`, snu:1496-1501)
    if (w->guess_mode == 1 && n >= 3 && dts[n - 1] == dts[n - 2]) {
      LAUNCH(ctx, k_axpby, cdiv((size_t)(nv + np), 256), 256, 0, 2.0, (const double *)w->x.p, -1.0,
             (const double *)w->xprev.p, w->xguess.p, (size_t)(nv + np));
      DNSB_CK(ctx, cudaMemcpyAsync(w->xprev.p, w->x.p, (nv + np) * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
      DNSB_CK(ctx, cudaMemcpyAsync(w->x.p, w->xguess.p, (nv + np) * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
      DNSB_CK(ctx, cudaMemcpyAsync(w->xprev.p, w->x.p, (nv + np) * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    s->expect_its = 0;
    rc = solver_solve_dev(s, w->b.p, w->x.p, tol, maxit, false);
    if (rc) return rc;
    DNSB_CK(ctx, cudaMemcpyAsync(w->v.p, w->x.p, nv * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    LAUNCH(ctx, k_extract_p, cdiv((size_t)np, 256), 256, 0, (const double *)w->x.p, w->p.p, nv, np, 1, -1.0 / dt);
    // "current" side about the new state
    LAUNCH(ctx, k_scatter_inner, cdiv((size_t)nv, 256), 256, 0, (const double *)w->v.p, w->inv.p, w->vfull.p, nv, 1);
    rc = cnsweep_conv(w, w->vfull.p, picard != 0, w->nvc.p, w->fc.p);
    if (rc) return rc;
    DNSB_CK(ctx, cudaMemcpyAsync(w->vtraj.p + (size_t)n * nvf, w->vfull.p, nvf * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    DNSB_CK(ctx, cudaMemcpyAsync(w->ptraj.p + (size_t)n * np, w->p.p, np * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    // update norm  dt (v - lin)^T M (v - lin)
    LAUNCH(ctx, k_diff_inner, cdiv(nv, 256), 256, 0, (const double *)w->v.p, lin_n, (const int *)w->inv.p, w->dvec.p, nv);
    spmm_dev(ctx, w->M, nullptr, w->dvec.p, nullptr, w->mdv.p, 1, 1.0, 0.0);
    LAUNCH(ctx, k_dot1, rcn.nblocks, rcn.threads, rcn.smem, (const double *)w->dvec.p, (const double *)w->mdv.p, nv, 1, rcn.rpb, w->npart.p);
    LAUNCH(ctx, k_reduce_partials2, 1, 1024, 0, (const double *)w->npart.p, rcn.nblocks, 1, w->nout.p);
    double hn = 0.0;
    DNSB_CK(ctx, cudaMemcpyAsync(&hn, w->nout.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
    norm_acc += dt * hn;
  }
  DNSB_CK(ctx, cudaMemcpyAsync(vtraj, w->vtraj.p, (size_t)(nsteps + 1) * nvf * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaMemcpyAsync(ptraj, w->ptraj.p, (size_t)(nsteps + 1) * np * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  if (upd_norm) *upd_norm = norm_acc;
  if (iters_total) *iters_total = s->stat_iters - its0;
  DNSB_CK(ctx, cudaGetLastError());
  if (solver_relmax(s, false, &w->max_relres)) return -1;
  w->unconverged = s->stat_unconverged - unc0;
  if (w->unconverged > 0) {
    char msg[200];
    snprintf(msg, sizeof msg, "FGMRES stopped at maxit=%d above tol=%.1e in %lld of the %d step solves of this sweep "
             "(largest final relative residual %.3e)", maxit, tol, w->unconverged, nsteps, w->max_relres);
    ctx->fail(msg, __FILE__, __LINE__);
    return DNSB_E_NOT_CONVERGED;
  }
  return 0;
}

extern "C" int dnsb_cnsweep_set_guess(dnsb_cnsweep *w, int mode) {
  if (!w) return -2;
  DNSB_REQUIRE(w->ctx, mode == 0 || mode == 1, "guess mode: 0 (previous solution) or 1 (extrapolation)");
  w->guess_mode = mode;
  return 0;
}

extern "C" int dnsb_cnsweep_stats(dnsb_cnsweep *w, double *max_relres, long long *unconverged) {
  if (!w) return -2;
  if (max_relres) *max_relres = w->max_relres;
  if (unconverged) *unconverged = w->unconverged;
  return 0;
}

// z = P^-1 r on host vectors: the preconditioner alone (tests compare it with
// a numpy restatement of the same hierarchy)
extern "C" int dnsb_solver_apply_prec(dnsb_solver *s, const double *r, double *z) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, r && z, "null arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t ntb = (size_t)s->ntot * s->nb;
  DNSB_CK(ctx, s->sb.alloc(ntb));
  DNSB_CK(ctx, s->sx.alloc(ntb));
  DNSB_CK(ctx, cudaMemcpyAsync(s->sb.p, r, ntb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  DNSB_CK(ctx, cudaMemsetAsync(s->sx.p, 0, ntb * sizeof(double), ctx->stream));
  if (apply_prec(s, s->sb.p, s->sx.p)) return -1;
  DNSB_CK(ctx, cudaMemcpyAsync(z, s->sx.p, ntb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int dnsb_solver_set_prec_mode(dnsb_solver *s, int block_diagonal) {
  if (!s) return -2;
  s->prec_diag = block_diagonal ? 1 : 0;
  solver_drop_graphs(s);
  return 0;
}

// y = K x for the solver's saddle-point matrix, host vectors (ntot x nb)
extern "C" int dnsb_solver_apply_k(dnsb_solver *s, const double *x, double *y) {
  if (!s) return -2;
  dnsb_ctx *ctx = s->ctx;
  DNSB_REQUIRE(ctx, x && y, "null arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t ntb = (size_t)s->ntot * s->nb;
  DNSB_CK(ctx, s->sb.alloc(ntb));
  DNSB_CK(ctx, s->sx.alloc(ntb));
  DNSB_CK(ctx, cudaMemcpyAsync(s->sb.p, x, ntb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  spmm_dev(ctx, s->K.get(), s->has_coef ? s->coef.p : nullptr, s->sb.p, nullptr, s->sx.p, s->nb, 1.0, 0.0);
  DNSB_CK(ctx, cudaMemcpyAsync(y, s->sx.p, ntb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// ===========================================================================
// IMEX time stepper
// ===========================================================================
struct dnsb_imex {
  dnsb_ctx *ctx = nullptr;
  unsigned long long mesh_hash = 0;
  int scheme = 0, nb = 1, nv = 0, np = 0, nvf = 0, nbc = 0;
  double dt = 0;
  dnsb_csr *M = nullptr, *A = nullptr, *J = nullptr, *JT = nullptr;
  std::unique_ptr<dnsb_csr> Rm;   // CNAB rhs operator  M - dt/2*A_m
  dnsb_solver *sl = nullptr, *sp = nullptr, *sc = nullptr;
  DBuf<double> nu, coefR, coefA;   // nb
  DBuf<int> inv, bcinds;
  DBuf<double> bcvals, fv, fp;
  // forcing
  int nk = 0, ntimes = 0;
  long long force_t0 = 0;   // time level of useries[0]
  DBuf<double> Bk, useries;
  // state
  DBuf<double> v, vprev, p, vfull, cfull, nfc_c, nfc_o, nfc_t, tmp, b, x;
  // solution / rhs history for the initial guesses
  // guess <= 1: ring of the last two solutions (xh).  guess >= 2: projection
  // space: pairs (xq_i, bq_i) with K xq_i = bq_i (computed, not assumed) and
  // orthonormal bq_i, at most `hist_len` of them; ring `xh` of the last
  // `keep` raw solutions for the rebuild when the space is full
  int hist_len = 0, hist_cnt = 0, hist_pos = 0, hist_mode = 0;
  int pcnt = 0, pkeep = 0;
  DBuf<double> xh, bq, xq, gr, partialh, x0, pw0, pw1, pd0, pd1, pinv, normpart, normout;
  DBuf<double> ptri, py, pgsum;   // implicit form of the projection space (see imex_guess)
  bool proj_t = false;
  double last_relres = 0;   // max over ALL solves of the last run (every member, Heun solves included)
  long long run_iters = 0, run_solves = 0, run_unconverged = 0;
  // snapshots: device store (device row order; input of the Gram matrix) and
  // a pinned host mirror in OUTPUT row order, filled by async D2H copies on
  // a second stream while the integration goes on
  DBuf<double> snaps;
  int nsnap = 0, snap_cap = 0;
  DBuf<int> outmap;            // nv + np: output row of device row i
  bool has_outmap = false;
  static const int NSTAGE = 4;
  DBuf<double> stage[NSTAGE];  // gathered [v; p] in output order
  cudaEvent_t ev_ready[NSTAGE] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_free[NSTAGE] = {nullptr, nullptr, nullptr, nullptr};
  bool stage_busy[NSTAGE] = {false, false, false, false};
  cudaStream_t cstream = nullptr;
  PinnedBuf<double> h_snaps;   // h_cap snapshots
  int h_cap = 0;
  bool host_mirror = true;
  long long step = 0;   // steps done so far
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // device time of the last run
  float last_run_ms = 0.f;
  bool have_state = false;
  bool p_stale = false;
  // output functionals (dnsb_imex_set_outputs / dnsb_imex_set_force): ny linear rows + 2 force rows per
  // time level.  The rows are kept on the host as given (either call rebuilds the device arrays), the
  // record (levels, ny + 2, nb) grows at the start of a run like the snapshot store.
  int ny = 0;
  std::vector<int> cv_ptr, cv_idx, cp_ptr, cp_idx, fm_ptr, fm_idx, fa_ptr, fa_idx, fj_ptr, fj_idx, fdofs;
  std::vector<double> cv_val, cp_val, fm_val, fa_val, fj_val;
  double fbc[2] = {0.0, 0.0};
  DBuf<int> o_vptr, o_vidx, o_pptr, o_pidx, o_fptr, o_fdofs;
  DBuf<double> o_w1, o_w2, o_wp, o_fbc, o_csave, o_rec;
  int nlev = 0, lev_cap = 0;
  long long csave_level = -1;   // time level n whose Phi^T c(V_n) is in o_csave (-1: none)
  // per-member blow-up guard (dnsb_imex_set_member_guard): trip level of every member (-1: live) on the
  // host and on the device, and the frozen trip states (v, p lanes) of the retired members.  The device
  // arrays exist from the first retirement on; nretired == 0 launches nothing of this machinery.
  bool member_guard = false;
  std::vector<int> trip;
  int nretired = 0;
  DBuf<int> d_trip;
  DBuf<double> trip_v, trip_p;
  // in-loop statistics (dnsb_imex_set_statistics): Welford accumulators of the time levels st_first..st_last,
  // members fastest: st_v (nvf: mean of V in full numbering), st_cov (3 x nnodes: co-moments uu, vv, uv of
  // the two components of a node), st_pm / st_p2 (np: mean and M2 of p), st_c (nv: mean of c(V)[inv])
  bool stats_on = false;
  long long st_first = 0, st_last = -1;
  DBuf<double> st_v, st_cov, st_pm, st_p2, st_c;
  bool outputs_on() const { return ny > 0 || !fdofs.empty(); }
  ~dnsb_imex() {
    cudaStreamSynchronize(ctx->stream);   // no buffer is freed under a running kernel or copy
    if (cstream) { cudaStreamSynchronize(cstream); cudaStreamDestroy(cstream); }
    for (int q = 0; q < NSTAGE; ++q) {
      if (ev_ready[q]) cudaEventDestroy(ev_ready[q]);
      if (ev_free[q]) cudaEventDestroy(ev_free[q]);
    }
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

extern "C" int dnsb_imex_create(dnsb_ctx *ctx, int scheme, int nb, double dt,
                                dnsb_csr *mmat, dnsb_csr *amat, dnsb_csr *jmat,
                                dnsb_csr *jtmat, const double *nu,
                                const int32_t *invinds, int nv, int nbc,
                                const int32_t *bcinds, const double *bcvals,
                                const double *fv, const double *fp, dnsb_imex **out) {
  if (out) *out = nullptr;
  if (!ctx) return -2;
  DNSB_REQUIRE(ctx, out && mmat && amat && jmat && jtmat && nu && invinds, "null arguments");
  DNSB_REQUIRE(ctx, scheme >= 0 && scheme <= 2, "scheme must be 0 (CNAB), 1 (SBDF2) or 2 (IMEX Euler)");
  DNSB_REQUIRE(ctx, ctx->ncell > 0, "set the mesh first");
  DNSB_REQUIRE(ctx, nb >= 1 && dt > 0, "bad nb/dt");
  DNSB_REQUIRE(ctx, mmat->nrows == nv && amat->nrows == nv && jmat->ncols == nv, "matrix sizes vs nv");
  DNSB_REQUIRE(ctx, mmat->nnz == amat->nnz, "M and A must share one pattern");
  DNSB_REQUIRE(ctx, amat->has2, "amat needs vals2 = a0 (nu-independent stiffness)");
  for (int k = 0; k < mmat->nnz; ++k)
    DNSB_REQUIRE(ctx, mmat->h_indices[k] == amat->h_indices[k], "M and A must share one pattern");
  const int nvf = 2 * ctx->nnodes;
  for (int i = 0; i < nv; ++i)
    DNSB_REQUIRE(ctx, invinds[i] >= 0 && invinds[i] < nvf, "invinds out of range");
  for (int i = 0; i < nbc; ++i)
    DNSB_REQUIRE(ctx, bcinds[i] >= 0 && bcinds[i] < nvf, "bcinds out of range");
  DNSB_CK(ctx, dnsb_enter(ctx));
  std::unique_ptr<dnsb_imex> e(new (std::nothrow) dnsb_imex());
  DNSB_REQUIRE(ctx, e != nullptr, "out of host memory");
  e->ctx = ctx; e->scheme = scheme; e->nb = nb; e->dt = dt;
  e->trip.assign(nb, -1);
  e->mesh_hash = ctx->mesh_hash;
  e->nv = nv; e->np = jmat->nrows; e->nvf = nvf; e->nbc = nbc;
  e->M = mmat; e->A = amat; e->J = jmat; e->JT = jtmat;
  DNSB_CK(ctx, e->nu.upload(nu, nb, ctx->stream));
  std::vector<double> cr(nb);
  for (int m = 0; m < nb; ++m) cr[m] = -0.5 * dt * nu[m];
  DNSB_CK(ctx, e->coefR.upload(cr.data(), nb, ctx->stream));
  DNSB_CK(ctx, e->inv.upload(invinds, nv, ctx->stream));
  if (nbc > 0) {
    DNSB_CK(ctx, e->bcinds.upload(bcinds, nbc, ctx->stream));
    DNSB_CK(ctx, e->bcvals.upload(bcvals, nbc, ctx->stream));
  }
  std::vector<double> zero(std::max(nv, e->np), 0.0);
  DNSB_CK(ctx, e->fv.upload(fv ? fv : zero.data(), nv, ctx->stream));
  DNSB_CK(ctx, e->fp.upload(fp ? fp : zero.data(), e->np, ctx->stream));
  if (scheme == 0) {
    // R = M - dt/2*arob  (vals1),  a0 (vals2) with coef -dt/2*nu_m
    std::vector<double> r1(mmat->nnz);
    for (int k = 0; k < mmat->nnz; ++k) r1[k] = mmat->h_v1[k] - 0.5 * dt * amat->h_v1[k];
    int rc = csr_build(ctx, nv, nv, mmat->h_indptr.data(), mmat->h_indices.data(), r1.data(),
                       amat->h_v2.data(), e->Rm);
    if (rc) return rc;
    // the right-hand side product R v of every step through the staged tile kernel as well (bit-identical)
    if (nb == TILE_NB) { rc = tile_setup(ctx, e->Rm.get()); if (rc) return rc; }
  }
  const size_t nvb = (size_t)nv * nb, npb = (size_t)e->np * nb, nfb = (size_t)nvf * nb;
  DNSB_CK(ctx, e->v.alloc(nvb)); DNSB_CK(ctx, e->vprev.alloc(nvb));
  DNSB_CK(ctx, e->p.alloc(npb));
  DNSB_CK(ctx, e->vfull.alloc(nfb)); DNSB_CK(ctx, e->cfull.alloc(nfb));
  DNSB_CK(ctx, e->nfc_c.alloc(nvb)); DNSB_CK(ctx, e->nfc_o.alloc(nvb));
  DNSB_CK(ctx, e->nfc_t.alloc(nvb)); DNSB_CK(ctx, e->tmp.alloc(nvb));
  DNSB_CK(ctx, e->b.alloc(nvb + npb)); DNSB_CK(ctx, e->x.alloc(nvb + npb));
  DNSB_CK(ctx, cudaEventCreate(&e->ev0));
  DNSB_CK(ctx, cudaEventCreate(&e->ev1));
  DNSB_CK(ctx, e->vfull.zero(ctx->stream));
  if (nbc > 0)
    LAUNCH(ctx, k_set_bcs, cdiv((size_t)nbc * nb, 256), 256, 0, e->bcinds.p, e->bcvals.p,
           e->vfull.p, nbc, nb);
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  *out = e.release();
  return 0;
}

extern "C" void dnsb_imex_destroy(dnsb_imex *e) {
  if (!e) return;
  dnsb_enter(e->ctx);
  delete e;
}

extern "C" int dnsb_imex_set_solvers(dnsb_imex *e, dnsb_solver *loop, dnsb_solver *pred,
                                     dnsb_solver *corr) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, loop != nullptr, "loop solver required");
  for (dnsb_solver *s : {loop, pred, corr})
    if (s) DNSB_REQUIRE(ctx, s->nv == e->nv && s->np == e->np && s->nb == e->nb, "solver shape mismatch");
  if (e->scheme != 2) DNSB_REQUIRE(ctx, pred && corr, "CNAB/SBDF2 need the Heun solvers");
  e->sl = loop; e->sp = pred; e->sc = corr;
  return 0;
}

extern "C" int dnsb_imex_set_forcing(dnsb_imex *e, int nk, const double *bvecs,
                                     int ntimes, const double *useries) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, nk >= 0 && (nk == 0 || (bvecs && useries && ntimes >= 1)), "bad forcing");
  DNSB_CK(ctx, dnsb_enter(ctx));
  e->nk = nk; e->ntimes = ntimes;
  e->force_t0 = e->have_state ? e->step : 0;   // series starts at the current time level
  if (nk > 0) {
    DNSB_CK(ctx, e->Bk.upload(bvecs, (size_t)e->nv * nk, ctx->stream));
    DNSB_CK(ctx, e->useries.upload(useries, (size_t)ntimes * nk * e->nb, ctx->stream));
  }
  return 0;
}

extern "C" int dnsb_imex_set_state(dnsb_imex *e, const double *v0, const double *p0) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, v0 != nullptr, "null v0");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t nvb = (size_t)e->nv * e->nb, npb = (size_t)e->np * e->nb;
  DNSB_CK(ctx, cudaMemcpyAsync(e->v.p, v0, nvb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (p0)
    DNSB_CK(ctx, cudaMemcpyAsync(e->p.p, p0, npb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  else
    DNSB_CK(ctx, e->p.zero(ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  e->step = 0; e->hist_cnt = 0; e->hist_pos = 0; e->nsnap = 0; e->pcnt = 0;
  e->force_t0 = 0;
  e->nlev = 0; e->csave_level = -1;
  e->trip.assign(e->nb, -1); e->nretired = 0;   // every member is live again
  e->st_first = 0; e->st_last = -1;
  e->have_state = true;
  e->p_stale = false;
  return 0;
}

// nfc = -c(vfull)[inv] for the current inner velocity `v`
static int imex_nonl(dnsb_imex *e, const double *v, double *nfc) {
  dnsb_ctx *ctx = e->ctx;
  const size_t nvb = (size_t)e->nv * e->nb;
  LAUNCH(ctx, k_scatter_inner, cdiv(nvb, 256), 256, 0, v, e->inv.p, e->vfull.p, e->nv, e->nb);
  if (g_conv_colours) {
    int rc = convvec_dev(ctx, e->vfull.p, nullptr, e->cfull.p, e->nb);
    if (rc) return rc;
    LAUNCH(ctx, k_gather_neg, cdiv(nvb, 256), 256, 0, e->cfull.p, e->inv.p, nfc, e->nv, e->nb);
    return 0;
  }
  return convvec_dev(ctx, e->vfull.p, nullptr, nfc, e->nb, e->inv.p, e->nv, -1.0);
}

static const double *useries_at(dnsb_imex *e, long long n) {
  if (e->nk == 0) return nullptr;
  long long k = std::min<long long>(std::max<long long>(n - e->force_t0, 0), e->ntimes - 1);
  return e->useries.p + (size_t)k * e->nk * e->nb;
}

// p = -q/dt from the last saddle solution, if it is newer than e->p
static void imex_refresh_p(dnsb_imex *e) {
  if (!e->p_stale) return;
  const size_t npb = (size_t)e->np * e->nb;
  LAUNCH(e->ctx, k_extract_p, cdiv(npb, 256), 256, 0, e->x.p, e->p.p, e->nv, e->np, e->nb,
         -1.0 / e->dt);
  e->p_stale = false;
}

// out[map[i], m] = x[i, m]  (map == null: identity)
// copy != null: copy[t] = x[t] as well (the device-side trajectory store, same pass)
__global__ void k_scatter_rows(const double *__restrict__ x, const int *__restrict__ map,
                               double *__restrict__ out, int n, int nb, double *__restrict__ copy) {
  dnsb_pdl_entry();
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)n * nb) return;
  const int i = (int)(t / nb), m = (int)(t % nb);
  const int o = map ? map[i] : i;
  const double v = x[t];
  out[(size_t)o * nb + m] = v;
  if (copy) copy[t] = v;
}

// ---- per-member blow-up guard: the lanes of retired members ----------------
// trip[m] is the time level at which member m was retired, -1 while it is live.  Members are the fastest
// index of every vector, so lane m of a vector of n rows is x[i*nb + m].
// tv / tp lane m = v / p lane m for the members retired at `level`: their frozen trip state
__global__ void k_retire_take(const double *__restrict__ v, const double *__restrict__ p, double *__restrict__ tv,
                              double *__restrict__ tp, size_t nvb, size_t npb, int nb, const int *__restrict__ trip,
                              long long level) {
  dnsb_pdl_entry();
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nvb + npb) return;
  const size_t u = t < nvb ? t : t - nvb;
  if (trip[u % nb] != level) return;
  if (t < nvb) tv[u] = v[u]; else tp[u] = p[u];
}
// zero the retired lanes of the right-hand side b and the initial guess x (ntb each): such a lane enters
// FGMRES with b = 0 and x = 0 and is done at iteration 0, whatever its history buffers hold
__global__ void k_retire_zero(double *__restrict__ b, double *__restrict__ x, size_t ntb, int nb,
                              const int *__restrict__ trip) {
  dnsb_pdl_entry();
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntb || trip[t % nb] < 0) return;
  b[t] = 0.0;
  x[t] = 0.0;
}
// NaN in the lanes of the members retired before `level`, in a record of that level (x, and y if not null)
__global__ void k_retire_nan(double *__restrict__ x, double *__restrict__ y, size_t n, int nb,
                             const int *__restrict__ trip, long long level) {
  dnsb_pdl_entry();
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int tl = trip[t % nb];
  if (tl < 0 || level <= tl) return;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  x[t] = nan;
  if (y) y[t] = nan;
}
static int retire_nan(dnsb_imex *e, double *x, double *y, size_t n, long long level) {
  if (e->nretired == 0) return 0;
  LAUNCH(e->ctx, k_retire_nan, cdiv(n, 256), 256, 0, x, y, n, e->nb, (const int *)e->d_trip.p, level);
  return 0;
}

// fold time level `level` into the in-loop statistics (defined with its kernel at the end of the file, after
// every other kernel: ptxas then emits the SASS of all the others exactly as without it)
static int imex_stats(dnsb_imex *e, long long level, const double *nfc);

// pinned host mirror with room for `cap` snapshots (contents are kept)
static int imex_reserve_host(dnsb_imex *e, int cap) {
  dnsb_ctx *ctx = e->ctx;
  if (cap <= e->h_cap) return 0;
  const size_t ntb = (size_t)(e->nv + e->np) * e->nb;
  PinnedBuf<double> nh;
  DNSB_CK(ctx, nh.alloc((size_t)cap * ntb));
  if (e->h_snaps.p) {
    if (e->cstream) DNSB_CK(ctx, cudaStreamSynchronize(e->cstream));
    memcpy(nh.p, e->h_snaps.p, (size_t)std::min(e->nsnap, e->h_cap) * ntb * sizeof(double));
  }
  e->h_snaps = std::move(nh);
  e->h_cap = cap;
  return 0;
}

// snapshot = [v (nv*nb); p (np*nb)]: D2D into the device store and, in output
// row order, through a staging ring to the pinned host mirror (copy stream)
static int imex_snapshot(dnsb_imex *e) {
  dnsb_ctx *ctx = e->ctx;
  if (e->nsnap >= e->snap_cap) return 0;
  const size_t nvb = (size_t)e->nv * e->nb, npb = (size_t)e->np * e->nb, ntb = nvb + npb;
  imex_refresh_p(e);
  double *dst = e->snaps.p + (size_t)e->nsnap * ntb;
  const bool mirror = e->host_mirror && e->nsnap < e->h_cap;
  if (!mirror) {
    DNSB_CK(ctx, cudaMemcpyAsync(dst, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    DNSB_CK(ctx, cudaMemcpyAsync(dst + nvb, e->p.p, npb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    int rc = retire_nan(e, dst, nullptr, ntb, e->step);
    if (rc) return rc;
  }
  if (mirror) {   // the un-permuting kernels below fill the device-side store in the same pass
    const int q = e->nsnap % dnsb_imex::NSTAGE;
    if (e->stage_busy[q]) DNSB_CK(ctx, cudaStreamWaitEvent(ctx->stream, e->ev_free[q], 0));
    const int *mv = e->has_outmap ? e->outmap.p : nullptr;
    const int *mp = e->has_outmap ? e->outmap.p + e->nv : nullptr;
    LAUNCH(ctx, k_scatter_rows, cdiv(nvb, 256), 256, 0, (const double *)e->v.p, mv, e->stage[q].p, e->nv, e->nb, dst);
    LAUNCH(ctx, k_scatter_rows, cdiv(npb, 256), 256, 0, (const double *)e->p.p, mp, e->stage[q].p + nvb, e->np, e->nb,
           dst + nvb);
    int rc = retire_nan(e, dst, e->stage[q].p, ntb, e->step);
    if (rc) return rc;
    DNSB_CK(ctx, cudaEventRecord(e->ev_ready[q], ctx->stream));
    DNSB_CK(ctx, cudaStreamWaitEvent(e->cstream, e->ev_ready[q], 0));
    DNSB_CK(ctx, cudaMemcpyAsync(e->h_snaps.p + (size_t)e->nsnap * ntb, e->stage[q].p, ntb * sizeof(double),
                                 cudaMemcpyDeviceToHost, e->cstream));
    DNSB_CK(ctx, cudaEventRecord(e->ev_free[q], e->cstream));
    e->stage_busy[q] = true;
  }
  e->nsnap++;
  return 0;
}

// ---- output functionals ---------------------------------------------------
// Row r of the (ny + 2) x nb values of one time level n:
//   r < ny:      y_r = sum_k w1[k] vn[k] + ps sum_k wp[k] pn[k]                         (Cv v_n + Cp p_n)
//   r = ny + c:  F_c = rdt sum_k w1[k] (vn - vp)[k] + nu_m (1/2 sum_k w2[k] (vn + vp)[k] + fbc[c])
//                      - ps sum_k wp[k] pn[k] + 3/2 cc - 1/2 csave[c]
// the CNAB residual tested with the indicator of component c of the force dofs (residual_checks.get_imex_res):
// w1 = Phi^T M[:, inv], w2 = Phi^T A0[:, inv], wp = Phi^T JT, fbc = Phi^T A0[:, bc] u_bc, vp = v_{n-1}, and
// cc = Phi^T c(V_{n-1}) summed from the element buffer E of K1a through the node -> cell lists (as
// k_conv_gather does) or read from the full vector cfull (coloured K1a).  csave[c] holds Phi^T c(V_{n-2}) and
// receives cc.  fvalid = 0: the force is NaN (no earlier level to difference against); out == null: only
// csave is written (Heun start).  Block <-> (row, 32 members), lane <-> member: a warp reads 32 members of one
// column; warp w takes the terms w, w + OUT_WARPS, ... and the warps' sums are added in warp order, so the
// summation order is fixed and the result bit-reproducible.  The rows are short (a force row of cylinder_4:
// ~800 velocity, ~190 pressure terms, ~190 dofs): the kernel is bound by the latency of the dependent index ->
// value loads, hence many warps per row and unrolled loops (several loads in flight per warp).
#define OUT_WARPS 32
__global__ void __launch_bounds__(OUT_WARPS * 32)
k_imex_outputs(int ny, int row0, const int *__restrict__ vptr, const int *__restrict__ vidx,
               const double *__restrict__ w1, const double *__restrict__ w2, const int *__restrict__ pptr,
               const int *__restrict__ pidx, const double *__restrict__ wp, const int *__restrict__ fptr,
               const int *__restrict__ fdofs, const int *__restrict__ n2c_ptr, const int *__restrict__ n2c_idx,
               const double *__restrict__ E, const double *__restrict__ cfull, const double *__restrict__ vn,
               const double *__restrict__ vp, const double *__restrict__ pn, double ps, double rdt,
               const double *__restrict__ nu, const double *__restrict__ fbc, int fvalid, double *csave,
               double *__restrict__ out, int nb) {
  dnsb_pdl_entry();
  __shared__ double red[4][OUT_WARPS][32];
  const int r = row0 + blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int m = blockIdx.y * 32 + lane;
  const bool frow = r >= ny, act = m < nb;
  const bool conv = frow && (E != nullptr || cfull != nullptr);
  const bool sums = out != nullptr && (!frow || fvalid);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  if (act && sums) {
    if (frow) {
#pragma unroll 4
      for (int k = vptr[r] + w; k < vptr[r + 1]; k += OUT_WARPS) {
        const size_t o = (size_t)vidx[k] * nb + m;
        const double a = vn[o], b = vp[o];
        s0 += w1[k] * (a - b);
        s1 += w2[k] * (a + b);
      }
    } else {
#pragma unroll 4
      for (int k = vptr[r] + w; k < vptr[r + 1]; k += OUT_WARPS) s0 += w1[k] * vn[(size_t)vidx[k] * nb + m];
    }
#pragma unroll 4
    for (int k = pptr[r] + w; k < pptr[r + 1]; k += OUT_WARPS) s2 += wp[k] * pn[(size_t)pidx[k] * nb + m];
  }
  const int c = r - ny;
  if (act && conv) {
#pragma unroll 2
    for (int q = fptr[c] + w; q < fptr[c + 1]; q += OUT_WARPS) {
      const int dof = fdofs[q];
      if (cfull) {
        s3 += cfull[(size_t)dof * nb + m];
      } else {
        const int node = dof >> 1;
        double s = 0.0;
        for (int k = n2c_ptr[node]; k < n2c_ptr[node + 1]; ++k) s += E[((size_t)n2c_idx[k] * 2 + c) * nb + m];
        s3 += s;
      }
    }
  }
  red[0][w][lane] = s0; red[1][w][lane] = s1; red[2][w][lane] = s2; red[3][w][lane] = s3;
  __syncthreads();
  if (w != 0 || !act) return;
  double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
  for (int q = 0; q < OUT_WARPS; ++q) {
    t0 += red[0][q][lane]; t1 += red[1][q][lane]; t2 += red[2][q][lane]; t3 += red[3][q][lane];
  }
  if (out) {
    double val;
    if (!frow) val = t0 + ps * t2;
    else if (!fvalid) val = __longlong_as_double(0x7ff8000000000000ll);   // NaN
    else val = rdt * t0 + nu[m] * (0.5 * t1 + fbc[c]) - ps * t2 + 1.5 * t3 - 0.5 * csave[(size_t)c * nb + m];
    out[(size_t)r * nb + m] = val;
  }
  if (conv) csave[(size_t)c * nb + m] = t3;
}

// one launch of k_imex_outputs.  out_level: record the level into the next slot (vn, vp, pn, ps as in the
// kernel; vp may be null when the force is not valid); false: only capture Phi^T c of the convection the
// element buffer / cfull holds now (the caller says which level that is).  conv_level >= 0: the convection
// source holds c(V_{conv_level}), which the force of level conv_level + 1 needs together with the saved
// term of level conv_level - 1.
static int imex_outputs(dnsb_imex *e, bool out_level, const double *vn, const double *vp, const double *pn,
                        double ps, long long conv_level, long long level) {
  dnsb_ctx *ctx = e->ctx;
  const int nb = e->nb;
  const bool force = !e->fdofs.empty() && conv_level >= 0;
  const double *E = force && !g_conv_colours ? e->ctx->elem.p : nullptr;
  const double *cf = force && g_conv_colours ? e->cfull.p : nullptr;
  const int fvalid = force && out_level && e->csave_level == conv_level - 1 && vp != nullptr ? 1 : 0;
  const int row0 = out_level ? 0 : e->ny;
  const int nrows = out_level ? e->ny + 2 : 2;
  if (!out_level && !force) return 0;
  double *out = out_level ? e->o_rec.p + (size_t)e->nlev * (e->ny + 2) * nb : nullptr;
  LAUNCH(ctx, k_imex_outputs, dim3(nrows, cdiv(nb, 32)), OUT_WARPS * 32, 0, e->ny, row0,
         (const int *)e->o_vptr.p, (const int *)e->o_vidx.p, (const double *)e->o_w1.p, (const double *)e->o_w2.p,
         (const int *)e->o_pptr.p, (const int *)e->o_pidx.p, (const double *)e->o_wp.p, (const int *)e->o_fptr.p,
         (const int *)e->o_fdofs.p, (const int *)ctx->n2c_ptr.p, (const int *)ctx->n2c_idx.p, E, cf, vn, vp, pn, ps,
         1.0 / e->dt, (const double *)e->nu.p, (const double *)e->o_fbc.p, fvalid, e->o_csave.p, out, nb);
  if (force) e->csave_level = conv_level;
  if (out_level) {
    int rc = retire_nan(e, out, nullptr, (size_t)(e->ny + 2) * nb, level);   // `level` is that of the record
    if (rc) return rc;
    e->nlev++;
  }
  return 0;
}

// ---- initial guesses ------------------------------------------------------
// guess 0: previous solution; 1: linear extrapolation 2x_n - x_{n-1};
// L >= 2: residual-minimising projection onto the span of up to L earlier
// solutions of the same matrix K (Fischer 1998).  The space is kept as pairs
// (xq_i, bq_i) with K xq_i = bq_i and orthonormal bq_i, so that
//   x0 = sum_i <bq_i, b> xq_i   minimises |b - K x0| over the span.
// Unlike Fischer's recurrence the image of a new direction is COMPUTED
// (one SpMM) and orthogonalised twice (CGS2), with the same coefficients
// applied to the direction: the pairs stay consistent to round-off however
// small the new information is.  On cylinder_4, dt = 1/2048, eight pairs put
// the initial residual at ~1e-11 |b| (previous solution: 1e-3, linear
// extrapolation: 4e-6): the FGMRES then needs 1-3 iterations instead of 20.
// Implicit form (DNSB_PROJ_T=1, default): only the images bq_i are orthonormalised; the directions stay
// as they were handed in (D_i) and a small upper-triangular factor per member records the combination,
//   xq_j = sum_{i<=j} T[i][j] D_i,   x0 = sum_i (T c)_i D_i,   c = bq^T b.
// Every Gram-Schmidt pass over the xq side disappears (a third of the vector reads of proj_add).
// y[i] = sum_{j=i..k-1} T[i][j] c[j]
__global__ void k_proj_tri_apply(const double *__restrict__ T, const double *__restrict__ c,
                                 double *__restrict__ y, int k, int L, int nb) {
  dnsb_pdl_entry();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k * nb) return;
  const int i = t / nb, m = t % nb;
  double s = 0.0;
  for (int j = i; j < k; ++j) s += T[((size_t)i * L + j) * nb + m] * c[(size_t)j * nb + m];
  y[t] = s;
}
// column k of T after the direction D_k was cleaned with the coefficients g (sum over the passes) and
// normalised with inv:  T[i][k] = -inv * sum_{j=i..k-1} T[i][j] g[j],  T[k][k] = inv
__global__ void k_proj_tri_column(double *__restrict__ T, const double *__restrict__ g,
                                  const double *__restrict__ inv, int k, int L, int nb) {
  dnsb_pdl_entry();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (k + 1) * nb) return;
  const int i = t / nb, m = t % nb;
  if (i == k) { T[((size_t)k * L + k) * nb + m] = inv[m]; return; }
  double s = 0.0;
  for (int j = i; j < k; ++j) s += T[((size_t)i * L + j) * nb + m] * g[(size_t)j * nb + m];
  T[((size_t)i * L + k) * nb + m] = -inv[m] * s;
}
// x = x0 = sum_i y[i,m] D_i   (the guess and the copy the new direction is measured from, one pass)
__global__ void k_proj_guess(const double *__restrict__ D, size_t dstride, int nvec, const double *__restrict__ y,
                             double *__restrict__ x, double *__restrict__ x0, size_t n, int nb) {
  dnsb_pdl_entry();
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * nb) return;
  const int m = (int)(idx % nb);
  double s = 0.0;
  for (int i = 0; i < nvec; ++i) s += y[(size_t)i * nb + m] * D[(size_t)i * dstride + idx];
  x[idx] = s;
  x0[idx] = s;
}
// d = x - x0 and keep = x  (new direction + the ring of raw solutions, one pass)
__global__ void k_proj_dir(const double *__restrict__ x, const double *__restrict__ x0, double *__restrict__ d,
                           double *__restrict__ keep, size_t n) {
  dnsb_pdl_entry();
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const double v = x[idx];
  d[idx] = v - x0[idx];
  keep[idx] = v;
}
static int imex_guess(dnsb_imex *e, int guess, double *x) {
  dnsb_ctx *ctx = e->ctx;
  const int nb = e->nb;
  const int ntot = e->nv + e->np;
  const size_t ntb = (size_t)ntot * nb;
  const int L = e->hist_len;
  if (guess <= 1) {
    if (e->hist_cnt == 0) return 1;   // caller supplies the default guess
    const int last = (e->hist_pos + L - 1) % L;
    const double *xl = e->xh.p + (size_t)last * ntb;
    if (guess == 0 || e->hist_cnt == 1) {
      DNSB_CK(ctx, cudaMemcpyAsync(x, xl, ntb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
      const int prev = (e->hist_pos + L - 2) % L;
      LAUNCH(ctx, k_axpby, cdiv(ntb, 256), 256, 0, 2.0, xl, -1.0,
             (const double *)(e->xh.p + (size_t)prev * ntb), x, ntb);
    }
    return 0;
  }
  if (e->pcnt == 0) return 1;
  RedCfg rc = red_cfg(ctx, ntot, nb);
  mdot_dev(ctx, rc, e->bq.p, ntb, e->pcnt, e->b.p, ntot, nb, e->partialh.p, e->gr.p);
  const double *cf = e->gr.p;
  if (e->proj_t) {
    LAUNCH(ctx, k_proj_tri_apply, cdiv((size_t)e->pcnt * nb, 128), 128, 0, (const double *)e->ptri.p,
           (const double *)e->gr.p, e->py.p, e->pcnt, L, nb);
    cf = e->py.p;
  }
  // writes the guess and its copy x0 (imex_push_history measures the new direction from it)
  LAUNCH(ctx, k_proj_guess, cdiv(ntb, 256), 256, 0, (const double *)e->xq.p, ntb, e->pcnt, cf, x, e->x0.p,
         (size_t)ntot, nb);
  return 2;
}

// inv[m] = 1/sqrt(n2[m]) if n2[m] > eps*ref[m] else 0
__global__ void k_inv_norm(const double *__restrict__ n2, const double *__restrict__ ref,
                           double *__restrict__ inv, int nb, double eps) {
  dnsb_pdl_entry();
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= nb) return;
  const double v = n2[m];
  inv[m] = (v > eps * ref[m] && v > 0.0) ? 1.0 / sqrt(v) : 0.0;
}

// append the direction d (ntb, destroyed) to the projection space; `npass`
// Gram-Schmidt passes: the image of a correction x - x0 is orthogonal to the
// space already (up to the solver tolerance), one pass cleans it; a raw
// solution (rebuild) lies almost inside the space and needs two
static int proj_add(dnsb_imex *e, double *d, int npass) {
  dnsb_ctx *ctx = e->ctx;
  const int nb = e->nb, ntot = e->nv + e->np;
  const size_t ntb = (size_t)ntot * nb;
  dnsb_solver *sl = e->sl;
  const double *coef = sl->has_coef ? sl->coef.p : nullptr;
  RedCfg rc = red_cfg(ctx, ntot, nb);
  double *w = e->pw0.p, *w2 = e->pw1.p, *d2 = e->pd1.p;
  spmm_dev(ctx, sl->K.get(), coef, d, nullptr, w, nb, 1.0, 0.0);
  const int k = e->pcnt;
  // |K d|^2 before the orthogonalisation (reference for the breakdown test)
  for (int pass = 0; pass < npass && k > 0; ++pass) {
    mdot_dev(ctx, rc, e->bq.p, ntb, k, w, ntot, nb, e->partialh.p, e->gr.p);
    if (pass == 0)
      DNSB_CK(ctx, cudaMemcpyAsync(e->normout.p, e->gr.p + (size_t)k * nb, nb * sizeof(double),
                                   cudaMemcpyDeviceToDevice, ctx->stream));
    gs_update_dev(ctx, rc, e->bq.p, ntb, k, e->gr.p, w, w2, ntot, nb, e->normpart.p);
    if (e->proj_t) {
      if (pass == 0)
        DNSB_CK(ctx, cudaMemcpyAsync(e->pgsum.p, e->gr.p, (size_t)k * nb * sizeof(double),
                                     cudaMemcpyDeviceToDevice, ctx->stream));
      else
        LAUNCH(ctx, k_axpby, cdiv((size_t)k * nb, 256), 256, 0, 1.0, (const double *)e->pgsum.p, 1.0,
               (const double *)e->gr.p, e->pgsum.p, (size_t)k * nb);
    } else {
      gs_update_dev(ctx, rc, e->xq.p, ntb, k, e->gr.p, d, d2, ntot, nb, e->partialh.p);
      std::swap(d, d2);
    }
    std::swap(w, w2);
  }
  if (k == 0) {
    LAUNCH(ctx, k_dot1, rc.nblocks, rc.threads, rc.smem, (const double *)w, (const double *)w, ntot, nb,
           rc.rpb, e->normpart.p);
  }
  // |w|^2 of the orthogonalised image
  LAUNCH(ctx, k_reduce_partials2, cdiv(nb, 32), 1024, 0, (const double *)e->normpart.p, rc.nblocks, nb,
         e->pinv.p + nb);
  if (k == 0)
    DNSB_CK(ctx, cudaMemcpyAsync(e->normout.p, e->pinv.p + nb, nb * sizeof(double),
                                 cudaMemcpyDeviceToDevice, ctx->stream));
  LAUNCH(ctx, k_inv_norm, cdiv(nb, 64), 64, 0, (const double *)(e->pinv.p + nb),
         (const double *)e->normout.p, e->pinv.p, nb, 1e-26);
  LAUNCH(ctx, k_scale_member, cdiv(ntb, 256), 256, 0, (const double *)w, (const double *)e->pinv.p,
         e->bq.p + (size_t)k * ntb, (size_t)ntot, nb);
  if (e->proj_t) {
    // the direction itself is the new column of D (the caller may have built it in place)
    if (d != e->xq.p + (size_t)k * ntb)
      DNSB_CK(ctx, cudaMemcpyAsync(e->xq.p + (size_t)k * ntb, d, ntb * sizeof(double), cudaMemcpyDeviceToDevice,
                                   ctx->stream));
    LAUNCH(ctx, k_proj_tri_column, cdiv((size_t)(k + 1) * nb, 128), 128, 0, e->ptri.p, (const double *)e->pgsum.p,
           (const double *)e->pinv.p, k, e->hist_len, nb);
  } else {
    LAUNCH(ctx, k_scale_member, cdiv(ntb, 256), 256, 0, (const double *)d, (const double *)e->pinv.p,
           e->xq.p + (size_t)k * ntb, (size_t)ntot, nb);
  }
  e->pcnt = k + 1;
  return 0;
}

static int imex_push_history(dnsb_imex *e, int guess) {
  dnsb_ctx *ctx = e->ctx;
  if (e->hist_len == 0) return 0;
  const int nb = e->nb;
  const int ntot = e->nv + e->np;
  const size_t ntb = (size_t)ntot * nb;
  if (guess <= 1) {
    const int s = e->hist_pos;
    DNSB_CK(ctx, cudaMemcpyAsync(e->xh.p + (size_t)s * ntb, e->x.p, ntb * sizeof(double),
                                 cudaMemcpyDeviceToDevice, ctx->stream));
    e->hist_pos = (s + 1) % e->hist_len;
    e->hist_cnt++;
    return 0;
  }
  // ring of raw solutions (for the rebuild)
  const int K = e->pkeep;
  double *keep = e->xh.p + (size_t)(e->hist_pos % K) * ntb;
  e->hist_pos++;
  e->hist_cnt++;
  if (e->pcnt > 0 && e->pcnt < e->hist_len) {
    // new direction: the correction x - x0, written in the same pass as the ring copy
    double *dir = e->proj_t ? e->xq.p + (size_t)e->pcnt * ntb : e->pd0.p;
    LAUNCH(ctx, k_proj_dir, cdiv(ntb, 256), 256, 0, (const double *)e->x.p, (const double *)e->x0.p, dir, keep, ntb);
    return proj_add(e, dir, 1);
  }
  DNSB_CK(ctx, cudaMemcpyAsync(keep, e->x.p, ntb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  if (e->pcnt == 0 && e->pcnt < e->hist_len) {
    // empty space: the solution itself
    double *dir = e->proj_t ? e->xq.p : e->pd0.p;
    DNSB_CK(ctx, cudaMemcpyAsync(dir, e->x.p, ntb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    return proj_add(e, dir, 2);
  }
  // space full: rebuild it from the last K raw solutions, oldest first
  e->pcnt = 0;
  const int have = std::min(K, e->hist_cnt);
  for (int q = have; q >= 1; --q) {
    const int slot = (e->hist_pos - q) % K;
    double *dir = e->proj_t ? e->xq.p + (size_t)e->pcnt * ntb : e->pd0.p;
    DNSB_CK(ctx, cudaMemcpyAsync(dir, e->xh.p + (size_t)slot * ntb, ntb * sizeof(double),
                                 cudaMemcpyDeviceToDevice, ctx->stream));
    int rc = proj_add(e, dir, 2);
    if (rc) return rc;
  }
  return 0;
}

// blow-up guard (time_int_utils.py:94-103) at the current time level: |v_m| > maxv or NaN?  Stop-all mode:
// *stop if any member fails.  Member mode: the live members that fail are retired (their v / p lanes are
// frozen into trip_v / trip_p, trip[m] = this level, *retired = true) and *stop only once none is left.
static int imex_blowup(dnsb_imex *e, const double *vc, double maxv, bool *stop, bool *retired) {
  dnsb_ctx *ctx = e->ctx;
  const int nb = e->nb;
  RedCfg rcn = red_cfg(ctx, e->nv, nb);
  LAUNCH(ctx, k_dot1, rcn.nblocks, rcn.threads, rcn.smem, vc, vc, e->nv, nb, rcn.rpb, e->normpart.p);
  LAUNCH(ctx, k_reduce_partials2, cdiv(nb, 32), 1024, 0, (const double *)e->normpart.p, rcn.nblocks, nb, e->normout.p);
  std::vector<double> hn(nb);
  DNSB_CK(ctx, cudaMemcpyAsync(hn.data(), e->normout.p, nb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  *stop = false;
  if (!e->member_guard) {
    for (int m = 0; m < nb; ++m)
      if (!(std::sqrt(hn[m]) <= maxv)) *stop = true;   // also catches NaN
    return 0;
  }
  int fresh = 0;
  for (int m = 0; m < nb; ++m)
    if (e->trip[m] < 0 && !(std::sqrt(hn[m]) <= maxv)) { e->trip[m] = (int)e->step; ++fresh; }
  if (fresh == 0) return 0;
  *retired = true;
  if (e->nretired == 0) {
    DNSB_CK(ctx, e->trip_v.alloc((size_t)e->nv * nb));
    DNSB_CK(ctx, e->trip_p.alloc((size_t)e->np * nb));
  }
  e->nretired += fresh;
  DNSB_CK(ctx, e->d_trip.upload(e->trip.data(), nb, ctx->stream));
  imex_refresh_p(e);
  const size_t nvb = (size_t)e->nv * nb, npb = (size_t)e->np * nb;
  LAUNCH(ctx, k_retire_take, cdiv(nvb + npb, 256), 256, 0, (const double *)e->v.p, (const double *)e->p.p,
         e->trip_v.p, e->trip_p.p, nvb, npb, nb, (const int *)e->d_trip.p, e->step);
  *stop = e->nretired == nb;
  return 0;
}

extern "C" int dnsb_imex_run(dnsb_imex *e, int nsteps, int snap_stride, double tol,
                             int maxit, int guess, double check_ff_maxv,
                             int ntimeslices, int *ffflag) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, e->have_state, "set the initial state first");
  DNSB_REQUIRE(ctx, e->mesh_hash == ctx->mesh_hash,
               "the mesh of the context is not the one this integrator was created on (dnsb_set_mesh)");
  DNSB_REQUIRE(ctx, e->sl != nullptr, "set the solvers first");
  DNSB_REQUIRE(ctx, nsteps >= 1 && tol > 0 && maxit >= 1 && guess >= 0 && guess <= 64, "bad run arguments");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int nb = e->nb, nv = e->nv, np = e->np;
  const size_t nvb = (size_t)nv * nb, npb = (size_t)np * nb, ntb = nvb + npb;
  const double dt = e->dt;
  if (ffflag) *ffflag = 0;
  // ---- history buffers -----------------------------------------------------
  {
    const int L = guess >= 2 ? guess : 2;
    const int mode = guess >= 2 ? 2 : 1;
    if (e->hist_len != L || e->hist_mode != mode) {
      e->hist_len = L; e->hist_cnt = 0; e->hist_pos = 0; e->hist_mode = mode; e->pcnt = 0;
      e->pkeep = g_pkeep > 0 ? std::max(1, std::min(g_pkeep, L)) : std::max(2, std::min(8, L / 2));
      DNSB_CK(ctx, e->xh.alloc(ntb * (mode == 2 ? e->pkeep : L)));
      DNSB_CK(ctx, e->xh.zero(ctx->stream));
      if (mode == 2) {
        RedCfg rc = red_cfg(ctx, nv + np, nb);
        DNSB_CK(ctx, e->bq.alloc(ntb * L));
        DNSB_CK(ctx, e->xq.alloc(ntb * L));
        DNSB_CK(ctx, e->gr.alloc((size_t)(L + 1) * nb));
        DNSB_CK(ctx, e->partialh.alloc((size_t)rc.nblocks * (L + 1) * nb));
        DNSB_CK(ctx, e->x0.alloc(ntb));
        DNSB_CK(ctx, e->pw0.alloc(ntb)); DNSB_CK(ctx, e->pw1.alloc(ntb));
        DNSB_CK(ctx, e->pd0.alloc(ntb)); DNSB_CK(ctx, e->pd1.alloc(ntb));
        DNSB_CK(ctx, e->pinv.alloc(2 * (size_t)nb));
        e->proj_t = g_proj_t != 0;
        if (e->proj_t) {
          DNSB_CK(ctx, e->ptri.alloc((size_t)L * L * nb));
          DNSB_CK(ctx, e->ptri.zero(ctx->stream));
          DNSB_CK(ctx, e->py.alloc((size_t)L * nb));
          DNSB_CK(ctx, e->pgsum.alloc((size_t)L * nb));
        }
      }
    }
  }
  {
    RedCfg rcn = red_cfg(ctx, nv, nb), rct = red_cfg(ctx, nv + np, nb);
    DNSB_CK(ctx, e->normpart.alloc((size_t)std::max(rcn.nblocks, rct.nblocks) * nb));
    DNSB_CK(ctx, e->normout.alloc(nb));
  }
  // ---- snapshots -----------------------------------------------------------
  if (snap_stride > 0) {
    const int need = e->nsnap + nsteps / snap_stride + 2;
    if (need > e->snap_cap) {
      DBuf<double> ns;
      DNSB_CK(ctx, ns.alloc((size_t)need * ntb));
      if (e->nsnap > 0)
        DNSB_CK(ctx, cudaMemcpyAsync(ns.p, e->snaps.p, (size_t)e->nsnap * ntb * sizeof(double),
                                     cudaMemcpyDeviceToDevice, ctx->stream));
      DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
      e->snaps = std::move(ns);
      e->snap_cap = need;
    }
    if (e->host_mirror) {
      if (!e->cstream) {
        DNSB_CK(ctx, cudaStreamCreateWithFlags(&e->cstream, cudaStreamNonBlocking));
        for (int q = 0; q < dnsb_imex::NSTAGE; ++q) {
          DNSB_CK(ctx, e->stage[q].alloc(ntb));
          DNSB_CK(ctx, cudaEventCreateWithFlags(&e->ev_ready[q], cudaEventDisableTiming));
          DNSB_CK(ctx, cudaEventCreateWithFlags(&e->ev_free[q], cudaEventDisableTiming));
        }
      }
      if (need > e->h_cap) { int rc = imex_reserve_host(e, need + need / 2); if (rc) return rc; }
    }
    if (e->step == 0) { int rc = imex_snapshot(e); if (rc) return rc; }
  }
  // ---- output functionals: room for this run's levels, the current one first if the record is empty --
  const bool outs = e->outputs_on();
  if (outs) {
    const size_t per = (size_t)(e->ny + 2) * nb;
    const int need = e->nlev + (e->nlev == 0 ? 1 : 0) + nsteps;
    if (need > e->lev_cap) {
      DBuf<double> nr;
      DNSB_CK(ctx, nr.alloc((size_t)need * per));
      if (e->nlev > 0)
        DNSB_CK(ctx, cudaMemcpyAsync(nr.p, e->o_rec.p, (size_t)e->nlev * per * sizeof(double),
                                     cudaMemcpyDeviceToDevice, ctx->stream));
      DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
      e->o_rec = std::move(nr);
      e->lev_cap = need;
    }
    if (e->nlev == 0) {
      imex_refresh_p(e);
      int rc = imex_outputs(e, true, e->v.p, nullptr, e->p.p, 1.0, -1, e->step);
      if (rc) return rc;
    }
  }
  const long long it0 = e->sl->stat_iters, ns0 = e->sl->stat_solves;
  dnsb_solver *const run_solvers[3] = {e->sl, e->sp, e->sc};
  long long unc0 = 0;
  for (dnsb_solver *sv : run_solvers)
    if (sv) {
      unc0 += sv->stat_unconverged;
      DNSB_CK(ctx, sv->grelmax.zero(ctx->stream));
    }
  DNSB_CK(ctx, cudaEventRecord(e->ev0, ctx->stream));
  int done = 0;
  // ======================= start-up (Heun) step =============================
  if (e->step == 0 && e->scheme != 2) {
    const double *u0 = useries_at(e, 0), *u1 = useries_at(e, 1);
    int rc = imex_nonl(e, e->v.p, e->nfc_c.p);                 // nfc(v0)
    if (rc) return rc;
    rc = imex_stats(e, 0, e->nfc_c.p);
    if (rc) return rc;
    if (outs && e->scheme == 0) {   // Phi^T c(V_0), before the predictor's convection overwrites it
      rc = imex_outputs(e, false, nullptr, nullptr, nullptr, 0.0, 0, 0);
      if (rc) return rc;
    }
    // predictor (IMEX Euler):  (M + dt A) tv = M v + dt f(t1) + dt nfc(v0)
    spmm_dev(ctx, e->M, nullptr, e->v.p, nullptr, e->b.p, nb, 1.0, 0.0);
    LAUNCH(ctx, k_rhs_combine, cdiv(nvb, 256), 256, 0, e->b.p, (const double *)e->nfc_c.p, dt,
           (const double *)nullptr, 0.0, (const double *)e->fv.p, dt, (const double *)e->Bk.p, e->nk,
           (const double *)nullptr, 0.0, u1, dt, nv, nb);
    LAUNCH(ctx, k_fill_rhsp, cdiv(npb, 256), 256, 0, e->b.p, e->fp.p, nv, np, nb);
    DNSB_CK(ctx, cudaMemcpyAsync(e->x.p, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    DNSB_CK(ctx, cudaMemsetAsync(e->x.p + nvb, 0, npb * sizeof(double), ctx->stream));
    e->sp->expect_its = 0;
    rc = solver_solve_dev(e->sp, e->b.p, e->x.p, tol, maxit, false);
    if (rc) return rc;
    // corrector:  M v1 = M v - dt/2 A (v + tv) + dt/2 (f0 + f1 + nfc(v0) + nfc(tv))
    rc = imex_nonl(e, e->x.p, e->nfc_t.p);                      // nfc(tv)
    if (rc) return rc;
    LAUNCH(ctx, k_axpby, cdiv(nvb, 256), 256, 0, 1.0, (const double *)e->v.p, 1.0,
           (const double *)e->x.p, e->tmp.p, nvb);
    spmm_dev(ctx, e->M, nullptr, e->v.p, nullptr, e->b.p, nb, 1.0, 0.0);
    spmm_dev(ctx, e->A, e->nu.p, e->tmp.p, e->b.p, e->b.p, nb, -0.5 * dt, 1.0);
    LAUNCH(ctx, k_rhs_combine, cdiv(nvb, 256), 256, 0, e->b.p, (const double *)e->nfc_c.p, 0.5 * dt,
           (const double *)e->nfc_t.p, 0.5 * dt, (const double *)e->fv.p, dt,
           (const double *)e->Bk.p, e->nk, u0, 0.5 * dt, u1, 0.5 * dt, nv, nb);
    LAUNCH(ctx, k_fill_rhsp, cdiv(npb, 256), 256, 0, e->b.p, e->fp.p, nv, np, nb);
    e->sc->expect_its = 0;
    rc = solver_solve_dev(e->sc, e->b.p, e->x.p, tol, maxit, false);
    if (rc) return rc;
    if (e->scheme == 1)
      DNSB_CK(ctx, cudaMemcpyAsync(e->vprev.p, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    DNSB_CK(ctx, cudaMemcpyAsync(e->v.p, e->x.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    e->p_stale = true;
    imex_refresh_p(e);
    e->step = 1;
    done = 1;
    if (outs) { rc = imex_outputs(e, true, e->v.p, nullptr, e->p.p, 1.0, -1, 1); if (rc) return rc; }
    if (snap_stride > 0 && e->step % snap_stride == 0) { rc = imex_snapshot(e); if (rc) return rc; }
    // nfc_c holds nfc(v0): it becomes nfc_o in the first loop step
  }
  // ======================= the time loop ====================================
  // blow-up guard at the start of each of the `ntimeslices` slices and of the
  // remainder slice (time_int_utils.py:94-103, 480-489)
  const int loopsteps = nsteps - done;
  const int lenofts = ntimeslices > 0 ? loopsteps / ntimeslices : 0;
  bool blown = false, retired = false;
  for (int it = 0; it < loopsteps; ++it) {
    if (ntimeslices > 0) {
      bool check = false;
      for (int k = 0; k <= ntimeslices; ++k)
        if (it == k * lenofts) check = true;
      if (check) {
        bool bad = false;
        int rcb = imex_blowup(e, e->scheme == 1 ? e->vprev.p : e->v.p, check_ff_maxv, &bad, &retired);
        if (rcb) return rcb;
        if (bad) { blown = true; break; }
      }
    }
    const long long n = e->step + 1;   // index of the new time level
    const double *uc = useries_at(e, n - 1), *un = useries_at(e, n);
    int rc;
    if (e->scheme == 0) {
      std::swap(e->nfc_o.p, e->nfc_c.p);
      rc = imex_nonl(e, e->v.p, e->nfc_c.p);
      if (rc) return rc;
      rc = imex_stats(e, n - 1, e->nfc_c.p);
      if (rc) return rc;
      spmm_dev(ctx, e->Rm.get(), e->coefR.p, e->v.p, nullptr, e->b.p, nb, 1.0, 0.0);
      LAUNCH(ctx, k_rhs_combine, cdiv(nvb, 256), 256, 0, e->b.p, (const double *)e->nfc_c.p, 1.5 * dt,
             (const double *)e->nfc_o.p, -0.5 * dt, (const double *)e->fv.p, dt,
             (const double *)e->Bk.p, e->nk, uc, 0.5 * dt, un, 0.5 * dt, nv, nb);
    } else if (e->scheme == 1) {
      std::swap(e->nfc_o.p, e->nfc_c.p);
      rc = imex_nonl(e, e->v.p, e->nfc_c.p);
      if (rc) return rc;
      rc = imex_stats(e, n - 1, e->nfc_c.p);
      if (rc) return rc;
      // rhs = 1/3 M (4 v_c - v_p) + 2/3 dt (2 nfc_c - nfc_p) + 2/3 dt f_n
      LAUNCH(ctx, k_axpby, cdiv(nvb, 256), 256, 0, 4.0 / 3.0, (const double *)e->v.p, -1.0 / 3.0,
             (const double *)e->vprev.p, e->tmp.p, nvb);
      spmm_dev(ctx, e->M, nullptr, e->tmp.p, nullptr, e->b.p, nb, 1.0, 0.0);
      LAUNCH(ctx, k_rhs_combine, cdiv(nvb, 256), 256, 0, e->b.p, (const double *)e->nfc_c.p,
             4.0 / 3.0 * dt, (const double *)e->nfc_o.p, -2.0 / 3.0 * dt, (const double *)e->fv.p,
             2.0 / 3.0 * dt, (const double *)e->Bk.p, e->nk, (const double *)nullptr, 0.0, un,
             2.0 / 3.0 * dt, nv, nb);
    } else {
      // IMEX Euler: (M + dt A) v+ = M v + dt (f(t+) + nfc(v))
      rc = imex_nonl(e, e->v.p, e->nfc_c.p);
      if (rc) return rc;
      rc = imex_stats(e, n - 1, e->nfc_c.p);
      if (rc) return rc;
      spmm_dev(ctx, e->M, nullptr, e->v.p, nullptr, e->b.p, nb, 1.0, 0.0);
      LAUNCH(ctx, k_rhs_combine, cdiv(nvb, 256), 256, 0, e->b.p, (const double *)e->nfc_c.p, dt,
             (const double *)nullptr, 0.0, (const double *)e->fv.p, dt, (const double *)e->Bk.p,
             e->nk, (const double *)nullptr, 0.0, un, dt, nv, nb);
    }
    LAUNCH(ctx, k_fill_rhsp, cdiv(npb, 256), 256, 0, e->b.p, e->fp.p, nv, np, nb);
    rc = imex_guess(e, guess, e->x.p);
    if (rc < 0) return rc;
    if (rc == 1) {   // no history yet: [v; q = -dt p]
      DNSB_CK(ctx, cudaMemcpyAsync(e->x.p, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
      LAUNCH(ctx, k_axpby, cdiv(npb, 256), 256, 0, -dt, (const double *)e->p.p, 0.0,
             (const double *)nullptr, e->x.p + nvb, npb);
    }
    if (e->nretired > 0)
      LAUNCH(ctx, k_retire_zero, cdiv(ntb, 256), 256, 0, e->b.p, e->x.p, ntb, nb, (const int *)e->d_trip.p);
    if (guess >= 2 && rc != 2)   // rc == 2: imex_guess wrote x0 itself
      DNSB_CK(ctx, cudaMemcpyAsync(e->x0.p, e->x.p, ntb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    rc = solver_solve_dev(e->sl, e->b.p, e->x.p, tol, maxit, false);
    if (rc) return rc;
    e->p_stale = true;
    if (outs) {   // level n from [v_n; q_n] = x, v_{n-1} = v and c(V_{n-1}) of this step's imex_nonl
      rc = imex_outputs(e, true, e->x.p, e->v.p, e->x.p + nvb, -1.0 / dt, e->scheme == 0 ? n - 1 : -1, n);
      if (rc) return rc;
    }
    rc = imex_push_history(e, guess);
    if (rc) return rc;
    if (e->scheme == 1)
      DNSB_CK(ctx, cudaMemcpyAsync(e->vprev.p, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    DNSB_CK(ctx, cudaMemcpyAsync(e->v.p, e->x.p, nvb * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    e->step = n;
    if (snap_stride > 0 && e->step % snap_stride == 0) { rc = imex_snapshot(e); if (rc) return rc; }
  }
  if (!blown && ntimeslices > 0 && ntimeslices * lenofts == loopsteps) {
    // the (empty) remainder slice still runs the guard once
    bool bad = false;
    int rcb = imex_blowup(e, e->scheme == 1 ? e->vprev.p : e->v.p, check_ff_maxv, &bad, &retired);
    if (rcb) return rcb;
    if (bad) blown = true;
  }
  if ((blown || retired) && ffflag) *ffflag = 1;
  imex_refresh_p(e);
  if (e->stats_on && e->st_last < e->step) {
    // the final level: its convection into e->tmp, which every step writes before it reads it
    int rc = imex_nonl(e, e->v.p, e->tmp.p);
    if (rc) return rc;
    rc = imex_stats(e, e->step, e->tmp.p);
    if (rc) return rc;
  }
  DNSB_CK(ctx, cudaEventRecord(e->ev1, ctx->stream));
  DNSB_CK(ctx, cudaEventSynchronize(e->ev1));
  if (snap_stride > 0 && e->cstream) DNSB_CK(ctx, cudaStreamSynchronize(e->cstream));
  DNSB_CK(ctx, cudaEventElapsedTime(&e->last_run_ms, e->ev0, e->ev1));
  // convergence of the run: the largest final relative residual over ALL
  // solves and members (the device keeps the running maximum), and the number
  // of solves that stopped at `maxit` above `tol`
  // (member mode: over the members live at the end of the run)
  int live_failed = 0;
  {
    double mx = 0.0;
    long long unc = -unc0;
    for (dnsb_solver *sv : run_solvers)
      if (sv) {
        std::vector<double> h;
        if (solver_relmax_members(sv, h)) return -1;
        for (int m = 0; m < nb; ++m) {
          if (e->member_guard && e->trip[m] >= 0) continue;
          const double r = h[m];
          if (mx == mx && !(r <= mx)) mx = r;   // NaN wins
          if (!(r <= tol)) ++live_failed;
        }
        unc += sv->stat_unconverged;
      }
    e->last_relres = mx;
    e->run_unconverged = unc;
  }
  e->run_iters = e->sl->stat_iters - it0;
  e->run_solves = e->sl->stat_solves - ns0;
  DNSB_CK(ctx, cudaGetLastError());
  if (e->member_guard) {
    // per-member verdict: a member retired in this run is forgiven its solves, a live one is not
    if (live_failed == 0) return 0;
    char msg[240];
    snprintf(msg, sizeof msg, "a member live at the end of the run has a final relative residual above tol=%.1e "
             "or a non-finite one (largest over the live members %.3e; FGMRES maxit=%d)", tol, e->last_relres,
             maxit);
    ctx->fail(msg, __FILE__, __LINE__);
    return DNSB_E_NOT_CONVERGED;
  }
  if (e->last_relres != e->last_relres && !blown) {
    // inf/NaN right-hand sides "converge" trivially (NaN compares false): a blown-up member with
    // the guard of time_int_utils.py:94-103 switched off (ntimeslices = 0) must not pass silently
    ctx->fail("a solve of this run had a non-finite residual: the state of at least one member has blown up "
              "(run with the blow-up guard, ntimeslices > 0, to get the reference's ffflag instead)",
              __FILE__, __LINE__);
    return DNSB_E_NOT_CONVERGED;
  }
  if (e->run_unconverged > 0 && !blown) {
    // the state is valid and can be read; the caller decides (the reference's
    // exact LU solve cannot fail this way, so the default is to refuse)
    char msg[200];
    snprintf(msg, sizeof msg, "FGMRES stopped at maxit=%d above tol=%.1e in %lld solve(s) of this run "
             "(largest final relative residual %.3e)", maxit, tol, e->run_unconverged, e->last_relres);
    ctx->fail(msg, __FILE__, __LINE__);
    return DNSB_E_NOT_CONVERGED;
  }
  return 0;
}

extern "C" int dnsb_imex_get_state(dnsb_imex *e, double *v, double *p) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t nvb = (size_t)e->nv * e->nb, npb = (size_t)e->np * e->nb;
  if (v) DNSB_CK(ctx, cudaMemcpyAsync(v, e->v.p, nvb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (p) DNSB_CK(ctx, cudaMemcpyAsync(p, e->p.p, npb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  if (e->nretired == 0) return 0;
  // retired members: their frozen trip state
  const int nb = e->nb;
  std::vector<double> tv(v ? nvb : 0), tp(p ? npb : 0);
  if (v) DNSB_CK(ctx, cudaMemcpyAsync(tv.data(), e->trip_v.p, nvb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (p) DNSB_CK(ctx, cudaMemcpyAsync(tp.data(), e->trip_p.p, npb * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  for (int m = 0; m < nb; ++m) {
    if (e->trip[m] < 0) continue;
    if (v) for (size_t i = 0; i < (size_t)e->nv; ++i) v[i * nb + m] = tv[i * nb + m];
    if (p) for (size_t i = 0; i < (size_t)e->np; ++i) p[i * nb + m] = tp[i * nb + m];
  }
  return 0;
}

extern "C" int dnsb_imex_set_member_guard(dnsb_imex *e, int on) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, on || e->nretired == 0,
               "members are retired: dnsb_imex_set_state makes them live before the stop-all guard can return");
  e->member_guard = on != 0;
  return 0;
}

extern "C" int dnsb_imex_member_status(dnsb_imex *e, int32_t *trip_level) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, trip_level != nullptr, "null output");
  for (int m = 0; m < e->nb; ++m) trip_level[m] = e->trip[m];
  return 0;
}

extern "C" int dnsb_imex_set_statistics(dnsb_imex *e, int on) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_CK(ctx, dnsb_enter(ctx));
  e->stats_on = false;
  if (!on) {
    for (DBuf<double> *b : {&e->st_v, &e->st_cov, &e->st_pm, &e->st_p2, &e->st_c}) b->release();
    return 0;
  }
  const size_t nb = e->nb, nnodes = e->nvf / 2;
  DNSB_CK(ctx, e->st_v.alloc((size_t)e->nvf * nb));
  DNSB_CK(ctx, e->st_cov.alloc(3 * nnodes * nb));
  DNSB_CK(ctx, e->st_pm.alloc((size_t)e->np * nb));
  DNSB_CK(ctx, e->st_p2.alloc((size_t)e->np * nb));
  DNSB_CK(ctx, e->st_c.alloc((size_t)e->nv * nb));
  e->stats_on = true;
  e->st_first = e->step; e->st_last = e->step - 1;
  return 0;
}

extern "C" int dnsb_imex_reset_statistics(dnsb_imex *e) {
  if (!e) return -2;
  DNSB_REQUIRE(e->ctx, e->stats_on, "statistics are off (dnsb_imex_set_statistics)");
  e->st_first = e->step; e->st_last = e->step - 1;
  return 0;
}

extern "C" int dnsb_imex_get_statistics(dnsb_imex *e, long long *first, long long *last, long long *count,
                                        double *v_mean, double *uvcov, double *p_mean, double *p_var,
                                        double *c_mean) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, e->stats_on, "statistics are off (dnsb_imex_set_statistics)");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int nb = e->nb, nnodes = e->nvf / 2;
  if (first) *first = e->st_first;
  if (last) *last = e->st_last;
  // levels of each member: a retired one stops at its trip level
  std::vector<long long> cnt(nb);
  const long long n = e->st_last - e->st_first + 1;
  for (int m = 0; m < nb; ++m)
    cnt[m] = e->trip[m] < 0 ? n : std::max(0LL, std::min(n, (long long)e->trip[m] - e->st_first + 1));
  if (count) for (int m = 0; m < nb; ++m) count[m] = cnt[m];
  struct Part { double *out; const DBuf<double> *src; size_t rows; bool moment; };
  const Part parts[] = {{v_mean, &e->st_v, (size_t)e->nvf, false}, {uvcov, &e->st_cov, 3 * (size_t)nnodes, true},
                        {p_mean, &e->st_pm, (size_t)e->np, false}, {p_var, &e->st_p2, (size_t)e->np, true},
                        {c_mean, &e->st_c, (size_t)e->nv, false}};
  for (const Part &q : parts)
    if (q.out)
      DNSB_CK(ctx, cudaMemcpyAsync(q.out, q.src->p, q.rows * nb * sizeof(double), cudaMemcpyDeviceToHost,
                                   ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  // co-moments -> population (co)variances; a member without levels is NaN
  const double nan = std::numeric_limits<double>::quiet_NaN();
  for (const Part &q : parts) {
    if (!q.out) continue;
    for (size_t i = 0; i < q.rows; ++i)
      for (int m = 0; m < nb; ++m) {
        double &x = q.out[i * nb + m];
        if (cnt[m] == 0) x = nan;
        else if (q.moment) x /= (double)cnt[m];
      }
  }
  return 0;
}

extern "C" int dnsb_imex_num_snapshots(dnsb_imex *e) { return e ? e->nsnap : -2; }

extern "C" int dnsb_imex_reset_snapshots(dnsb_imex *e) {
  if (!e) return -2;
  e->nsnap = 0;
  return 0;
}

extern "C" double dnsb_imex_last_run_ms(dnsb_imex *e) { return e ? (double)e->last_run_ms : -1.0; }

extern "C" int dnsb_imex_get_snapshots(dnsb_imex *e, double *out) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, out != nullptr, "null output");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const size_t ntb = (size_t)(e->nv + e->np) * e->nb;
  if (e->nsnap == 0) return 0;
  if (e->host_mirror && e->h_snaps.p && e->nsnap <= e->h_cap) {
    DNSB_CK(ctx, cudaStreamSynchronize(e->cstream));
    memcpy(out, e->h_snaps.p, (size_t)e->nsnap * ntb * sizeof(double));
    return 0;
  }
  DNSB_REQUIRE(ctx, !e->has_outmap, "host mirror disabled: no output order available");
  DNSB_CK(ctx, cudaMemcpyAsync(out, e->snaps.p, (size_t)e->nsnap * ntb * sizeof(double),
                               cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dnsb_imex_snapshots_host(dnsb_imex *e, const double **ptr, int *nsnap) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, ptr && nsnap, "null output");
  DNSB_REQUIRE(ctx, e->host_mirror, "host mirror disabled");
  if (e->cstream) DNSB_CK(ctx, cudaStreamSynchronize(e->cstream));
  *ptr = e->h_snaps.p;
  *nsnap = std::min(e->nsnap, e->h_cap);
  return 0;
}

extern "C" int dnsb_imex_set_output_order(dnsb_imex *e, const int32_t *vmap, const int32_t *pmap) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_CK(ctx, dnsb_enter(ctx));
  if (!vmap || !pmap) { e->has_outmap = false; return 0; }
  std::vector<int> mp((size_t)e->nv + e->np);
  std::vector<char> seen(std::max(e->nv, e->np));
  std::fill(seen.begin(), seen.end(), 0);
  for (int i = 0; i < e->nv; ++i) {
    DNSB_REQUIRE(ctx, vmap[i] >= 0 && vmap[i] < e->nv && !seen[vmap[i]], "vmap is not a permutation");
    seen[vmap[i]] = 1; mp[i] = vmap[i];
  }
  std::fill(seen.begin(), seen.end(), 0);
  for (int i = 0; i < e->np; ++i) {
    DNSB_REQUIRE(ctx, pmap[i] >= 0 && pmap[i] < e->np && !seen[pmap[i]], "pmap is not a permutation");
    seen[pmap[i]] = 1; mp[e->nv + i] = pmap[i];
  }
  DNSB_CK(ctx, e->outmap.upload(mp.data(), mp.size(), ctx->stream));
  e->has_outmap = true;
  return 0;
}

extern "C" int dnsb_imex_reserve_snapshots(dnsb_imex *e, int nsnap) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, nsnap >= 0, "bad count");
  DNSB_CK(ctx, dnsb_enter(ctx));
  return imex_reserve_host(e, nsnap);
}

// ---- output functionals: host side --------------------------------------------
static void rows_copy(const dnsb_csr *a, std::vector<int> &ptr, std::vector<int> &idx, std::vector<double> &val) {
  if (!a) { ptr.clear(); idx.clear(); val.clear(); return; }
  ptr = a->h_indptr; idx = a->h_indices; val = a->h_v1;
}

// device arrays of k_imex_outputs from the rows kept on the host: velocity rows (Cv | union of the
// patterns of Phi^T M and Phi^T A0), pressure rows (Cp | Phi^T JT), force dofs by component
static int outputs_upload(dnsb_imex *e) {
  dnsb_ctx *ctx = e->ctx;
  const int ny = e->ny;
  std::vector<int> vptr(1, 0), vidx, pptr(1, 0), pidx;
  std::vector<double> w1, w2, wp;
  for (int r = 0; r < ny; ++r) {
    if (!e->cv_ptr.empty())
      for (int k = e->cv_ptr[r]; k < e->cv_ptr[r + 1]; ++k) {
        vidx.push_back(e->cv_idx[k]); w1.push_back(e->cv_val[k]); w2.push_back(0.0);
      }
    vptr.push_back((int)vidx.size());
    if (!e->cp_ptr.empty())
      for (int k = e->cp_ptr[r]; k < e->cp_ptr[r + 1]; ++k) { pidx.push_back(e->cp_idx[k]); wp.push_back(e->cp_val[k]); }
    pptr.push_back((int)pidx.size());
  }
  const bool force = !e->fdofs.empty();
  std::vector<double> dm(force ? e->nv : 0), da(force ? e->nv : 0);
  std::vector<char> hit(force ? e->nv : 0);
  for (int c = 0; c < 2; ++c) {
    if (force) {
      std::fill(dm.begin(), dm.end(), 0.0); std::fill(da.begin(), da.end(), 0.0);
      std::fill(hit.begin(), hit.end(), 0);
      for (int k = e->fm_ptr[c]; k < e->fm_ptr[c + 1]; ++k) { dm[e->fm_idx[k]] += e->fm_val[k]; hit[e->fm_idx[k]] = 1; }
      for (int k = e->fa_ptr[c]; k < e->fa_ptr[c + 1]; ++k) { da[e->fa_idx[k]] += e->fa_val[k]; hit[e->fa_idx[k]] = 1; }
      for (int i = 0; i < e->nv; ++i)
        if (hit[i]) { vidx.push_back(i); w1.push_back(dm[i]); w2.push_back(da[i]); }
      for (int k = e->fj_ptr[c]; k < e->fj_ptr[c + 1]; ++k) { pidx.push_back(e->fj_idx[k]); wp.push_back(e->fj_val[k]); }
    }
    vptr.push_back((int)vidx.size());
    pptr.push_back((int)pidx.size());
  }
  // force dofs: unique, x components first, ascending
  std::vector<int> fd, fptr(3, 0);
  for (int c = 0; c < 2; ++c) {
    for (int d : e->fdofs) if ((d & 1) == c) fd.push_back(d);
    std::sort(fd.begin() + fptr[c], fd.end());
    fd.erase(std::unique(fd.begin() + fptr[c], fd.end()), fd.end());
    fptr[c + 1] = (int)fd.size();
  }
  // empty lists still get a valid pointer
  if (vidx.empty()) { vidx.push_back(0); w1.push_back(0.0); w2.push_back(0.0); }
  if (pidx.empty()) { pidx.push_back(0); wp.push_back(0.0); }
  if (fd.empty()) fd.push_back(0);
  DNSB_CK(ctx, e->o_vptr.upload(vptr.data(), vptr.size(), ctx->stream));
  DNSB_CK(ctx, e->o_vidx.upload(vidx.data(), vidx.size(), ctx->stream));
  DNSB_CK(ctx, e->o_w1.upload(w1.data(), w1.size(), ctx->stream));
  DNSB_CK(ctx, e->o_w2.upload(w2.data(), w2.size(), ctx->stream));
  DNSB_CK(ctx, e->o_pptr.upload(pptr.data(), pptr.size(), ctx->stream));
  DNSB_CK(ctx, e->o_pidx.upload(pidx.data(), pidx.size(), ctx->stream));
  DNSB_CK(ctx, e->o_wp.upload(wp.data(), wp.size(), ctx->stream));
  DNSB_CK(ctx, e->o_fptr.upload(fptr.data(), fptr.size(), ctx->stream));
  DNSB_CK(ctx, e->o_fdofs.upload(fd.data(), fd.size(), ctx->stream));
  DNSB_CK(ctx, e->o_fbc.upload(e->fbc, 2, ctx->stream));
  DNSB_CK(ctx, e->o_csave.alloc((size_t)2 * e->nb));
  // a new layout starts a new record
  e->nlev = 0; e->lev_cap = 0; e->o_rec.release();
  return 0;
}

extern "C" int dnsb_imex_set_outputs(dnsb_imex *e, dnsb_csr *cv, dnsb_csr *cp) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, !cv || cv->ncols == e->nv, "Cv must have nv columns (inner velocity)");
  DNSB_REQUIRE(ctx, !cp || cp->ncols == e->np, "Cp must have np columns (pressure)");
  DNSB_REQUIRE(ctx, !cv || !cp || cv->nrows == cp->nrows, "Cv and Cp must have the same number of rows");
  DNSB_CK(ctx, dnsb_enter(ctx));
  e->ny = cv ? cv->nrows : cp ? cp->nrows : 0;
  rows_copy(cv, e->cv_ptr, e->cv_idx, e->cv_val);
  rows_copy(cp, e->cp_ptr, e->cp_idx, e->cp_val);
  return outputs_upload(e);
}

extern "C" int dnsb_imex_set_force(dnsb_imex *e, int ndofs, const int32_t *dofs, dnsb_csr *fm, dnsb_csr *fa,
                                   dnsb_csr *fj, const double *fa_bc) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, ndofs >= 0, "bad number of force dofs");
  if (ndofs > 0) {
    DNSB_REQUIRE(ctx, e->scheme == 0,
                 "forces are the CNAB residual (scheme 0); SBDF2 / IMEX Euler have no force functional");
    DNSB_REQUIRE(ctx, dofs && fm && fa && fj && fa_bc, "null force arguments");
    DNSB_REQUIRE(ctx, fm->nrows == 2 && fm->ncols == e->nv, "Phi^T M must be 2 x nv");
    DNSB_REQUIRE(ctx, fa->nrows == 2 && fa->ncols == e->nv, "Phi^T A0 must be 2 x nv");
    DNSB_REQUIRE(ctx, fj->nrows == 2 && fj->ncols == e->np, "Phi^T JT must be 2 x np");
    for (int k = 0; k < ndofs; ++k)
      DNSB_REQUIRE(ctx, dofs[k] >= 0 && dofs[k] < e->nvf, "force dof out of range (full velocity numbering)");
  }
  DNSB_CK(ctx, dnsb_enter(ctx));
  if (ndofs > 0) e->fdofs.assign(dofs, dofs + ndofs); else e->fdofs.clear();
  rows_copy(ndofs ? fm : nullptr, e->fm_ptr, e->fm_idx, e->fm_val);
  rows_copy(ndofs ? fa : nullptr, e->fa_ptr, e->fa_idx, e->fa_val);
  rows_copy(ndofs ? fj : nullptr, e->fj_ptr, e->fj_idx, e->fj_val);
  e->fbc[0] = ndofs ? fa_bc[0] : 0.0;
  e->fbc[1] = ndofs ? fa_bc[1] : 0.0;
  e->csave_level = -1;
  return outputs_upload(e);
}

extern "C" int dnsb_imex_num_output_levels(dnsb_imex *e) { return e ? e->nlev : -2; }

extern "C" int dnsb_imex_reset_outputs(dnsb_imex *e) {
  if (!e) return -2;
  e->nlev = 0;
  return 0;
}

extern "C" int dnsb_imex_get_outputs(dnsb_imex *e, double *y, double *force) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int nb = e->nb, nr = e->ny + 2;
  if (e->nlev == 0) return 0;
  std::vector<double> h((size_t)e->nlev * nr * nb);
  DNSB_CK(ctx, cudaMemcpyAsync(h.data(), e->o_rec.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost,
                               ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  const size_t ly = (size_t)e->ny * nb, lf = (size_t)2 * nb;
  for (int l = 0; l < e->nlev; ++l) {
    const double *src = h.data() + (size_t)l * nr * nb;
    if (y && ly) memcpy(y + l * ly, src, ly * sizeof(double));
    if (force) memcpy(force + l * lf, src + ly, lf * sizeof(double));
  }
  return 0;
}

extern "C" int dnsb_imex_stats(dnsb_imex *e, long long *total_iters, long long *nsolves,
                               double *max_relres) {
  if (!e || !e->sl) return -2;
  if (total_iters) *total_iters = e->run_iters;
  if (nsolves) *nsolves = e->run_solves;
  if (max_relres) *max_relres = e->last_relres;
  return 0;
}

extern "C" long long dnsb_imex_unconverged(dnsb_imex *e) { return e ? e->run_unconverged : -2; }

// G[a,b] = sum_m sum_i X_a[i,m] * (M X_b)[i,m]; trip != null: only the members m with trip[m] < 0 (live)
__global__ void k_gram_partial(const double *__restrict__ X, size_t xstride,
                               const double *__restrict__ MX,
                               int ns, size_t nvb, double *__restrict__ partial,
                               const int *__restrict__ trip, int nb) {
  dnsb_pdl_entry();
  // block (a, b) pair over blockIdx.y; grid-stride chunks over blockIdx.x
  extern __shared__ double sred[];
  const int pair = blockIdx.y;
  const int a = pair / ns, b = pair % ns;
  const double *xa = X + (size_t)a * xstride, *mb = MX + (size_t)b * nvb;
  const size_t chunk = (nvb + gridDim.x - 1) / gridDim.x;
  const size_t i0 = (size_t)blockIdx.x * chunk, i1 = min(nvb, i0 + chunk);
  double acc = 0.0;
  if (trip) {
    for (size_t i = i0 + threadIdx.x; i < i1; i += blockDim.x)
      if (trip[i % nb] < 0) acc += xa[i] * mb[i];   // a retired lane may hold NaN: skipped, not weighted
  } else {
    for (size_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) acc += xa[i] * mb[i];
  }
  sred[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sred[threadIdx.x] += sred[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[(size_t)blockIdx.x * ns * ns + pair] = sred[0];
}

static int imex_gram_impl(dnsb_imex *e, double *g_dev);

extern "C" int dnsb_imex_gram(dnsb_imex *e, double *g) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, g != nullptr && e->nsnap > 0, "no snapshots / null output");
  DNSB_CK(ctx, dnsb_enter(ctx));
  DBuf<double> gd;
  DNSB_CK(ctx, gd.alloc((size_t)e->nsnap * e->nsnap));
  int rc = imex_gram_impl(e, gd.p);
  if (rc) return rc;
  DNSB_CK(ctx, cudaMemcpyAsync(g, gd.p, gd.n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int dnsb_imex_gram_dev(dnsb_imex *e, double *g_dev) { return imex_gram_impl(e, g_dev); }

static int imex_gram_impl(dnsb_imex *e, double *g_dev) {
  if (!e) return -2;
  dnsb_ctx *ctx = e->ctx;
  DNSB_REQUIRE(ctx, g_dev != nullptr && e->nsnap > 0, "no snapshots / null output");
  DNSB_CK(ctx, dnsb_enter(ctx));
  const int ns = e->nsnap, nb = e->nb;
  const size_t nvb = (size_t)e->nv * nb, ntb = (size_t)(e->nv + e->np) * nb;
  DBuf<double> MX, part;
  DNSB_CK(ctx, MX.alloc((size_t)ns * nvb));
  for (int a = 0; a < ns; ++a)
    spmm_dev(ctx, e->M, nullptr, e->snaps.p + (size_t)a * ntb, nullptr, MX.p + (size_t)a * nvb, nb, 1.0, 0.0);
  const int nchunks = 32;
  DNSB_CK(ctx, part.alloc((size_t)nchunks * ns * ns));
  LAUNCH(ctx, k_gram_partial, dim3(nchunks, ns * ns), 256, 256 * sizeof(double), e->snaps.p, ntb, MX.p, ns, nvb, part.p,
         e->nretired > 0 ? (const int *)e->d_trip.p : (const int *)nullptr, nb);
  LAUNCH(ctx, k_reduce_partials2, cdiv((size_t)ns * ns, 32), 1024, 0, (const double *)part.p, nchunks, ns * ns, g_dev);
  DNSB_CK(ctx, cudaStreamSynchronize(ctx->stream));
  DNSB_CK(ctx, cudaGetLastError());
  return 0;
}

// ---- in-loop statistics ----------------------------------------------------
// W consecutive members of row i of an (n, nb) array (W = 2: one 16-byte access)
template <int W>
__device__ __forceinline__ void st_load(const double *__restrict__ a, size_t i, int nb, int m, double (&r)[W]) {
  if constexpr (W == 2) {
    const double2 t = *reinterpret_cast<const double2 *>(a + i * nb + m);
    r[0] = t.x; r[1] = t.y;
  } else {
    r[0] = a[i * nb + m];
  }
}
template <int W>
__device__ __forceinline__ void st_store(double *__restrict__ a, size_t i, int nb, int m, const double (&r)[W]) {
  if constexpr (W == 2) *reinterpret_cast<double2 *>(a + i * nb + m) = make_double2(r[0], r[1]);
  else a[i * nb + m] = r[0];
}
// Fold one time level into the accumulators by an elementwise Welford update with the count k of that level
// (rk = 1/k; k == 1 writes the values themselves, so the buffers need no clearing).  One thread per W
// consecutive members of one row of the concatenated index space [nnodes nodes | nv inner dofs | np pressures]:
//   node i:   u = vfull[2i], v = vfull[2i+1]   ->  mean st_v[2i], st_v[2i+1]; co-moments cov[0|1|2][i] (uu, vv, uv)
//   inner j:  c = -nfc[j]                      ->  mean cm[j]
//   press. r: p = ps * pq[r]                   ->  mean pm[r], M2 p2[r]
// A member retired before `level` (0 <= trip[m] < level) keeps its values.  No reduction: the result does not
// depend on the launch shape and is bit-reproducible.
template <int W>
__global__ void k_imex_stats(const double *__restrict__ vfull, const double *__restrict__ nfc,
                             const double *__restrict__ pq, double ps, double *__restrict__ vm,
                             double *__restrict__ cov, double *__restrict__ cm, double *__restrict__ pm,
                             double *__restrict__ p2, int nnodes, int nv, int np, int nb,
                             const int *__restrict__ trip, long long level, bool first, double rk) {
  dnsb_pdl_entry();
  const int ng = nb / W;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)(nnodes + nv + np) * ng) return;
  const size_t row = t / ng;
  const int m = (int)(t % ng) * W;
  bool live[W];
  for (int w = 0; w < W; ++w) live[w] = !trip || trip[m + w] < 0 || trip[m + w] >= level;
  if (row < (size_t)nnodes) {
    const size_t i = row;
    double u[W], v[W], mu[W], mv[W], cuu[W], cvv[W], cuv[W];
    st_load<W>(vfull, 2 * i, nb, m, u);
    st_load<W>(vfull, 2 * i + 1, nb, m, v);
    st_load<W>(vm, 2 * i, nb, m, mu);
    st_load<W>(vm, 2 * i + 1, nb, m, mv);
    st_load<W>(cov, i, nb, m, cuu);
    st_load<W>(cov, nnodes + i, nb, m, cvv);
    st_load<W>(cov, 2 * (size_t)nnodes + i, nb, m, cuv);
    for (int w = 0; w < W; ++w) {
      if (!live[w]) continue;
      if (first) {
        mu[w] = u[w]; mv[w] = v[w]; cuu[w] = 0.0; cvv[w] = 0.0; cuv[w] = 0.0;
        continue;
      }
      const double du = u[w] - mu[w], dv = v[w] - mv[w];
      mu[w] += du * rk;
      mv[w] += dv * rk;
      const double eu = u[w] - mu[w], ev = v[w] - mv[w];
      cuu[w] += du * eu;
      cvv[w] += dv * ev;
      cuv[w] += du * ev;
    }
    st_store<W>(vm, 2 * i, nb, m, mu);
    st_store<W>(vm, 2 * i + 1, nb, m, mv);
    st_store<W>(cov, i, nb, m, cuu);
    st_store<W>(cov, nnodes + i, nb, m, cvv);
    st_store<W>(cov, 2 * (size_t)nnodes + i, nb, m, cuv);
  } else if (row < (size_t)(nnodes + nv)) {
    const size_t j = row - nnodes;
    double c[W], mc[W];
    st_load<W>(nfc, j, nb, m, c);
    st_load<W>(cm, j, nb, m, mc);
    for (int w = 0; w < W; ++w) {
      if (!live[w]) continue;
      mc[w] = first ? -c[w] : mc[w] + (-c[w] - mc[w]) * rk;
    }
    st_store<W>(cm, j, nb, m, mc);
  } else {
    const size_t r = row - nnodes - nv;
    double p[W], mp[W], q[W];
    st_load<W>(pq, r, nb, m, p);
    st_load<W>(pm, r, nb, m, mp);
    st_load<W>(p2, r, nb, m, q);
    for (int w = 0; w < W; ++w) {
      if (!live[w]) continue;
      const double x = ps * p[w];
      if (first) { mp[w] = x; q[w] = 0.0; continue; }
      const double d = x - mp[w];
      mp[w] += d * rk;
      q[w] += d * (x - mp[w]);
    }
    st_store<W>(pm, r, nb, m, mp);
    st_store<W>(p2, r, nb, m, q);
  }
}
// fold time level `level` into the statistics, once: vfull holds V_level (Dirichlet values included), nfc =
// -c(V_level)[inv], and its pressure is e->p, or -q/dt in x while e->p is stale (nothing between the solve and
// the next imex_guess writes x: imex_push_history / proj_add only read it)
static int imex_stats(dnsb_imex *e, long long level, const double *nfc) {
  if (!e->stats_on || level <= e->st_last) return 0;
  dnsb_ctx *ctx = e->ctx;
  const int nb = e->nb, nnodes = e->nvf / 2;
  const size_t nvb = (size_t)e->nv * nb;
  const double *pq = e->p_stale ? e->x.p + nvb : e->p.p;
  const double ps = e->p_stale ? -1.0 / e->dt : 1.0;
  const long long k = level - e->st_first + 1;
  const int *trip = e->nretired > 0 ? (const int *)e->d_trip.p : (const int *)nullptr;
  const bool pair = nb % 2 == 0;
  const size_t nthr = (size_t)(nnodes + e->nv + e->np) * (pair ? nb / 2 : nb);
  LAUNCH_IF(ctx, pair, k_imex_stats<2>, k_imex_stats<1>, cdiv(nthr, 256), 256, 0, (const double *)e->vfull.p, nfc,
            pq, ps, e->st_v.p, e->st_cov.p, e->st_c.p, e->st_pm.p, e->st_p2.p, nnodes, e->nv, e->np, nb, trip, level,
            k == 1, 1.0 / (double)k);
  e->st_last = level;
  return 0;
}

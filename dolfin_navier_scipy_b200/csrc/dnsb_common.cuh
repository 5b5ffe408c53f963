// dnsb_common.cuh -- context, device buffers, error handling (host side)
#pragma once
// L2 residency hints: 1 = the dense Schur inverse is read evict-first,
// 2 = also the Krylov basis in the Gram-Schmidt kernels
#ifndef DNSB_L2_HINTS
#define DNSB_L2_HINTS 2
#endif
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

struct dnsb_ctx;

// The programmatic launch attribute is only given to a kernel whose predecessor ON ITS STREAM is another
// kernel of this library: `griddepcontrol.wait` waits for prerequisite GRIDS, and a copy or memset that sits
// between two kernels is not one (measured: with the attribute on every launch, runs on the large mesh were
// no longer reproducible bit for bit).  Every other stream operation the library issues breaks the chain.
static cudaStream_t g_pdl_chain_stream = nullptr;   // stream whose last operation was one of our kernels
static inline void dnsb_pdl_break() { g_pdl_chain_stream = nullptr; }
#define cudaMemcpyAsync(...) (dnsb_pdl_break(), cudaMemcpyAsync(__VA_ARGS__))
#define cudaMemsetAsync(...) (dnsb_pdl_break(), cudaMemsetAsync(__VA_ARGS__))
#define cudaEventRecord(...) (dnsb_pdl_break(), cudaEventRecord(__VA_ARGS__))
#define cudaStreamWaitEvent(...) (dnsb_pdl_break(), cudaStreamWaitEvent(__VA_ARGS__))
#define cudaGraphLaunch(...) (dnsb_pdl_break(), cudaGraphLaunch(__VA_ARGS__))
#define cudaStreamBeginCapture(...) (dnsb_pdl_break(), cudaStreamBeginCapture(__VA_ARGS__))
#define cudaStreamEndCapture(...) (dnsb_pdl_break(), cudaStreamEndCapture(__VA_ARGS__))
#define cudaMemcpyToSymbol(...) (dnsb_pdl_break(), cudaMemcpyToSymbol(__VA_ARGS__))

// Programmatic dependent launch: every kernel of the library starts with this pair.  `launch_dependents`
// lets the NEXT kernel on the stream be scheduled once all CTAs of this one have started (its CTAs fill
// the SMs that drain during this kernel's tail, its launch latency is hidden), `wait` holds the kernel
// until every kernel it depends on has completed and flushed -- nothing is read before it, so the
// data dependencies are exactly those of plain stream order.  Both are no-ops for kernels launched
// without the programmatic-serialization attribute (DNSB_PDL=0).
__device__ __forceinline__ void dnsb_pdl_entry() {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 900
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

#define DNSB_CK(ctx, call)                                                    \
  do {                                                                        \
    cudaError_t e_ = (call);                                                  \
    if (e_ != cudaSuccess) {                                                  \
      (ctx)->fail(std::string(#call) + ": " + cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                  \
      return -1;                                                              \
    }                                                                         \
  } while (0)

#define DNSB_REQUIRE(ctx, cond, msg)                                          \
  do {                                                                        \
    if (!(cond)) {                                                            \
      (ctx)->fail(std::string(msg) + " [" #cond "]", __FILE__, __LINE__);     \
      return -2;                                                              \
    }                                                                         \
  } while (0)

// bytes held by live device [0] / pinned host [1] buffers of the whole process (dnsb_live_bytes)
static std::atomic<long long> g_live_bytes[2];

// Buffer of n T's in device memory (DBuf) or pinned host memory (PinnedBuf), owned by the object that
// holds it: the destructor frees it, a move hands it over, there are no copies.  Destructors do not
// throw, so nothing crosses the ABI as an exception.
template <class T, bool Pinned>
struct OwnedBuf {
  T *p = nullptr;
  size_t n = 0;
  OwnedBuf() = default;
  OwnedBuf(const OwnedBuf &) = delete;
  OwnedBuf &operator=(const OwnedBuf &) = delete;
  OwnedBuf(OwnedBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  OwnedBuf &operator=(OwnedBuf &&o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~OwnedBuf() { release(); }
  cudaError_t alloc(size_t count) {
    if (p && n == count) return cudaSuccess;   // reuse
    release();
    n = count;
    if (count == 0) return cudaSuccess;
    cudaError_t e = Pinned ? cudaMallocHost((void **)&p, count * sizeof(T)) : cudaMalloc((void **)&p, count * sizeof(T));
    if (e != cudaSuccess) { p = nullptr; n = 0; }
    else g_live_bytes[Pinned] += (long long)(count * sizeof(T));
    return e;
  }
  // upload / zero: device buffers
  cudaError_t upload(const T *h, size_t count, cudaStream_t s) {
    cudaError_t e = alloc(count);
    if (e != cudaSuccess || count == 0) return e;
    e = cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(s);   // host buffer is borrowed: finish now
  }
  cudaError_t zero(cudaStream_t s) {
    if (!n) return cudaSuccess;
    return cudaMemsetAsync(p, 0, n * sizeof(T), s);
  }
  void release() {
    if (p) {
      if (Pinned) cudaFreeHost(p); else cudaFree(p);
      g_live_bytes[Pinned] -= (long long)(n * sizeof(T));
    }
    p = nullptr;
    n = 0;
  }
};
template <class T> using DBuf = OwnedBuf<T, false>;
template <class T> using PinnedBuf = OwnedBuf<T, true>;

struct ProfRec {
  const char *name;
  cudaEvent_t e0, e1;
  long long work;   // caller-defined size of the launch (e.g. basis vectors of a Gram-Schmidt pass), or 0
};

struct dnsb_ctx {
  // per-kernel CUDA-event timing (dnsb_profile_begin/end); off by default
  bool prof = false;
  size_t prof_cap = 0;
  std::vector<ProfRec> recs;
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 0;
  int cc = 0;
  size_t mem_bytes = 0;
  std::string err;
  long long launches = 0;
  long long next_work = 0;   // recorded with the next profiled launch, then reset
  int pdl = 1;               // launch kernels with programmatic stream serialization (dnsb_pdl_entry)
  std::string pdl_only, pdl_skip;   // debugging: substring filters on the kernel name
  int sw[32] = {0};          // this context's tuning switches (DNSB_* environment at creation), see dnsb_enter

  // ---- mesh / convection data (cells permuted into colour order) ----------
  int ncell = 0, nnodes = 0, ncolours = 0;
  unsigned long long mesh_hash = 0;   // of the cell table + geometry: integrators check they run on their mesh
  DBuf<int> cn;          // 6*ncell, SoA: cn[k*ncell + c]
  DBuf<double> geom;     // 5*ncell, SoA
  DBuf<int> n2c_ptr, n2c_idx;   // node -> (permuted cell*6 + local node), ascending
  DBuf<double> elem;            // element vectors ncell*12*nb (K1a gather formulation)
  std::vector<int> colour_ptr;   // ncolours+1 offsets into the permuted cells
  std::vector<int> perm;         // permuted position -> original cell
  // fixed pattern of the P2 vector space + per-cell slots (144*ncell SoA)
  int cnnz = 0;
  DBuf<int> cindptr, cindices, cslots;
  DBuf<int> cslot_ptr, cslot_src;   // slot -> element contributions (K1b gather formulation)
  DBuf<double> en1, en2;            // element matrices 36*ncell / 144*ncell
  // staging buffers for the host-pointer entry points
  DBuf<double> stage_a, stage_b, stage_c, stage_d;

  void fail(const std::string &what, const char *file, int line) {
    char buf[64];
    snprintf(buf, sizeof buf, " (%s:%d)", file, line);
    err = what + buf;
  }
  void drop_recs() {
    for (ProfRec &r : recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    recs.clear();
  }
  ~dnsb_ctx() {   // the caller has made the device current (dnsb_enter)
    if (stream) cudaStreamSynchronize(stream);   // no buffer is freed under a running kernel
    drop_recs();
    if (stream) cudaStreamDestroy(stream);
  }
};

static inline unsigned int cdiv(size_t a, size_t b) {
  return (unsigned int)((a + b - 1) / b);
}

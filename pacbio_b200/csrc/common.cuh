// Shared host/device plumbing for the B200 mega-reads library: error handling, launch
// accounting, growable device buffers, event timers.  No torch types anywhere in this library.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "../../include/mega_reads_b200.h"

#define MR_FULL_MASK 0xffffffffu
constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs; persistent grids are sized in multiples of this

struct mr_workspace;
void mr_workspace_free(mr_workspace* ws);

struct mr_context {
  mr_workspace* ws = nullptr;          // scratch reused across batches (align.cu)
  int          device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // host -> device copies of staged batches (mr_stage_batch)
  cudaStream_t aux[9] = { };   // side streams for kernels that may overlap (chain tiers)
  cudaStream_t hi[9] = { };    // the same at the highest priority: the coords kernel that follows a tier's chaining kernel
  cudaEvent_t  ev[10] = { };
  cudaEvent_t  ev_hi[9] = { };
  std::string  err;
  uint64_t     launches = 0;
  bool         keep_taps = false;
  bool         chain_tables = false;   // constant tables of chain.cu uploaded to this device
  std::vector<std::pair<std::string, double>> timers;
  int          sm_count = kNumSMs;

  int fail(int code, const std::string& msg) { err = msg; return code; }
};

extern thread_local std::string g_mr_create_error;

#define MR_CUDA(ctx, call)                                                                     \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if(e__ != cudaSuccess) {                                                                   \
      char b__[512];                                                                           \
      snprintf(b__, sizeof(b__), "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return (ctx)->fail(e__ == cudaErrorMemoryAllocation ? MR_ENOMEM : MR_ECUDA, b__);       \
    }                                                                                          \
  } while(0)

#define MR_TRY(expr)              \
  do {                            \
    int rc__ = (expr);            \
    if(rc__ != MR_OK) return rc__; \
  } while(0)

// count + check a kernel launch
#define MR_LAUNCHED(ctx)                                      \
  do {                                                        \
    ++(ctx)->launches;                                        \
    MR_CUDA(ctx, cudaGetLastError());                         \
  } while(0)

// Growable device buffer.  Growth frees and reallocates (contents are NOT preserved).
struct dev_buf {
  void*  p = nullptr;
  size_t cap = 0;
  bool   owned = true;          // false: p points into another buffer (alias), never freed here
  ~dev_buf() { if(p && owned) cudaFree(p); }
  dev_buf() = default;
  dev_buf(const dev_buf&) = delete;
  dev_buf& operator=(const dev_buf&) = delete;
  int ensure(mr_context* ctx, size_t bytes) {
    if(bytes <= cap) return MR_OK;
    release();
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if(e != cudaSuccess) {
      cudaGetLastError();
      want = bytes;
      e = cudaMalloc(&p, want);
    }
    if(e != cudaSuccess) {
      cudaGetLastError();
      p = nullptr;
      char b[160];
      snprintf(b, sizeof(b), "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
      return ctx->fail(MR_ENOMEM, b);
    }
    cap = want;
    return MR_OK;
  }
  void release() { if(p && owned) cudaFree(p); p = nullptr; cap = 0; owned = true; }
  void alias(void* q, size_t bytes) { release(); p = q; cap = bytes; owned = false; }
  template<typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// pinned host buffer
struct pinned_buf {
  void*  p = nullptr;
  size_t cap = 0;
  ~pinned_buf() { if(p) cudaFreeHost(p); }
  pinned_buf() = default;
  pinned_buf(const pinned_buf&) = delete;
  pinned_buf& operator=(const pinned_buf&) = delete;
  int ensure(mr_context* ctx, size_t bytes) {
    if(bytes <= cap) return MR_OK;
    if(p) { cudaFreeHost(p); p = nullptr; cap = 0; }
    const size_t want = bytes + 64;
    cudaError_t e = cudaMallocHost(&p, want);
    if(e != cudaSuccess) { cudaGetLastError(); p = nullptr; return ctx->fail(MR_ENOMEM, "cudaMallocHost failed"); }
    cap = want;
    return MR_OK;
  }
  template<typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// scoped phase timer on the context stream (events; resolved at the next sync point)
struct phase_timer {
  mr_context* ctx;
  struct item { std::string name; cudaEvent_t a, b; };
  std::vector<item> items;
  explicit phase_timer(mr_context* c) : ctx(c) { }
  void begin(const char* name) {
    item it; it.name = name;
    cudaEventCreate(&it.a); cudaEventCreate(&it.b);
    cudaEventRecord(it.a, ctx->stream);
    items.push_back(it);
  }
  void end() { cudaEventRecord(items.back().b, ctx->stream); }
  void next(const char* name) { end(); begin(name); }
  // call after the stream has been synchronised
  void collect() {
    for(auto& it : items) {
      float ms = 0;
      if(cudaEventElapsedTime(&ms, it.a, it.b) != cudaSuccess) { cudaGetLastError(); ms = 0; }
      bool found = false;
      for(auto& t : ctx->timers) if(t.first == it.name) { t.second += ms * 1e-3; found = true; }
      if(!found) ctx->timers.push_back(std::make_pair(it.name, ms * 1e-3));
      cudaEventDestroy(it.a); cudaEventDestroy(it.b);
    }
    items.clear();
  }
  ~phase_timer() { for(auto& it : items) { cudaEventDestroy(it.a); cudaEventDestroy(it.b); } }
};

static inline unsigned div_up(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

// ---- small device helpers ----------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

// reverse the order of the 32 two-bit groups of a word (compact_dna stores base i at bits 2i,
// k-mer integers want the first base most significant)
__device__ __forceinline__ uint64_t reverse_pairs(uint64_t x) {
  x = __brevll(x);
  return ((x & 0x5555555555555555ULL) << 1) | ((x >> 1) & 0x5555555555555555ULL);
}

// ---- cp.async (LDGSTS): 8-byte copies global -> shared that do not pass through registers ----------
#ifdef __CUDACC__
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template<int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// ---- bulk asynchronous copies (the TMA engine's 1-D form, UBLKCP in SASS) completing on an mbarrier:
// one thread arms the barrier with the byte count and issues the copies, everybody waits on the
// barrier's phase.  Source, destination and size must be multiples of 16 bytes.
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(arrivals) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");     // visible to the async proxy
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* smem_dst, const void* gsrc, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while(!done);
}
#endif

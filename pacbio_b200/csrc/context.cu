// Context management for the C ABI: one context == one GPU == one stream.
#include "common.cuh"

#include <cstring>
#include <memory>

thread_local std::string g_mr_create_error;

extern "C" {

int mr_context_create(int device, mr_context** out) {
  if(!out) return MR_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if(e != cudaSuccess || count == 0) {
    cudaGetLastError();
    g_mr_create_error = std::string("no CUDA device available: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return MR_ENODEV;   // there is deliberately no CPU fallback
  }
  if(device < 0 || device >= count) { g_mr_create_error = "device ordinal out of range"; return MR_EINVAL; }
  e = cudaSetDevice(device);
  if(e != cudaSuccess) { g_mr_create_error = cudaGetErrorString(e); return MR_ECUDA; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if(e != cudaSuccess) { g_mr_create_error = cudaGetErrorString(e); return MR_ECUDA; }
  if(prop.major < 10) {
    g_mr_create_error = "this library is built for sm_100a (B200) only";
    return MR_ENODEV;
  }
  std::unique_ptr<mr_context> ctx(new mr_context);
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if(e != cudaSuccess) { g_mr_create_error = cudaGetErrorString(e); return MR_ECUDA; }
  {
    int least = 0, greatest = 0;
    if(cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) { cudaGetLastError(); greatest = 0; }
    for(auto& a : ctx->aux) if(cudaStreamCreateWithPriority(&a, cudaStreamNonBlocking, 0) != cudaSuccess) { cudaGetLastError(); a = nullptr; }
    for(auto& a : ctx->hi) if(cudaStreamCreateWithPriority(&a, cudaStreamNonBlocking, greatest) != cudaSuccess) { cudaGetLastError(); a = nullptr; }
  }
  cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  for(auto& v : ctx->ev) cudaEventCreateWithFlags(&v, cudaEventDisableTiming);
  for(auto& v : ctx->ev_hi) cudaEventCreateWithFlags(&v, cudaEventDisableTiming);
  *out = ctx.release();
  return MR_OK;
}

void mr_context_destroy(mr_context* ctx) {
  if(!ctx) return;
  cudaSetDevice(ctx->device);
  if(ctx->stream) cudaStreamSynchronize(ctx->stream);
  if(ctx->ws) mr_workspace_free(ctx->ws);
  for(auto& a : ctx->aux) if(a) { cudaStreamSynchronize(a); cudaStreamDestroy(a); }
  for(auto& a : ctx->hi) if(a) { cudaStreamSynchronize(a); cudaStreamDestroy(a); }
  for(auto& v : ctx->ev_hi) if(v) cudaEventDestroy(v);
  if(ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  for(auto& v : ctx->ev) if(v) cudaEventDestroy(v);
  if(ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* mr_last_error(const mr_context* ctx) { return ctx ? ctx->err.c_str() : g_mr_create_error.c_str(); }
int mr_context_device(const mr_context* ctx) { return ctx ? ctx->device : -1; }
uint64_t mr_context_launches(const mr_context* ctx) { return ctx ? ctx->launches : 0; }
void* mr_context_stream(mr_context* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int mr_context_sync(mr_context* ctx) {
  if(!ctx) return MR_EINVAL;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

int mr_context_timers(const mr_context* ctx, const char** names, double* seconds, int cap) {
  if(!ctx) return 0;
  int n = 0;
  for(const auto& t : ctx->timers) {
    if(n >= cap) break;
    if(names) names[n] = t.first.c_str();
    if(seconds) seconds[n] = t.second;
    ++n;
  }
  return n;
}

int mr_host_pin(mr_context* ctx, const void* p, size_t bytes) {
  if(!ctx || !p) return MR_EINVAL;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  MR_CUDA(ctx, cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterDefault));
  return MR_OK;
}

int mr_host_unpin(mr_context* ctx, const void* p) {
  if(!ctx || !p) return MR_EINVAL;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  MR_CUDA(ctx, cudaHostUnregister(const_cast<void*>(p)));
  return MR_OK;
}

int mr_context_keep_taps(mr_context* ctx, int on) {
  if(!ctx) return MR_EINVAL;
  ctx->keep_taps = on != 0;
  return MR_OK;
}

void mr_params_default(mr_params* p) {
  if(!p) return;
  memset(p, 0, sizeof(*p));
  p->stretch_factor = 1.3; p->stretch_constant = 10; p->stretch_cap = 10000.0; p->window_size = 1;
  p->forward = 1; p->max_match = 0; p->max_count = 5000; p->matching_mers = 0.0; p->matching_bases = 0.17;
  p->unitigs_k = 0; p->overlap_play = 1.3; p->errors = 3.0; p->bases = 0; p->run_graph = 1;
}

} // extern "C"

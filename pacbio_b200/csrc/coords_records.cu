// jf_aligner coords records on the device: print_coords (jf_aligner.cc:41-70) over the rows a batch left in the
// context's workspace, byte for byte what the host formatter (mrh::format_coords, host/host_common.cpp) prints.
//  1. measure: a thread per row sizes its line; a thread per read sizes the read's ">N name" header (compact format;
//     with -0 also for a read without rows).  Every read owns the slot before its rows, so slot read_coords[r] + r is
//     read r's header and slot row + r + 1 is that row's line.
//  2. scan: an exclusive scan of the slot lengths places every slot.
//  3. emit: a thread per slot writes it.  A line is ~150 bytes of numbers that depend on each other's lengths (the
//     three "%g" fields are rounded in a serial integer loop): a warp per line would leave 31 lanes idle through it.
// The text is copied into a pooled pinned slab.  The number formatters are records_common.hpp, shared with the host.
#include "align.cuh"
#include "records_common.hpp"

#include <cstring>
#include <memory>

struct mr_sr_names {
  int device = 0;
  uint32_t nseq = 0;
  dev_buf names, name_off, path_ids, path_off;
};

namespace {

struct crd_args {
  rows_args R;
  const char* sr_names; const uint64_t* sr_name_off;   // the super-reads' FASTA headers
  const uint32_t* path_ids; const uint64_t* path_off;  // their unitig paths, (id << 1) | (ori == 'R')
  uint32_t nseq;
  const char* names; const uint64_t* name_off;         // the reads' names
  int compact, zero_match;
  uint32_t* len;                                       // per slot (nrows + nreads)
  const uint64_t* off;
  char* text;
  unsigned long long* err;                             // smallest row whose super-read is not in the names
};

// Appends to a line: W = false only counts the bytes (the numbers are formatted into a scratch buffer), W = true
// writes them at `out`.
template<bool W> struct sink {
  char* out;
  uint32_t n = 0;
  char tmp[mrfmt::kGeneralMax + 8];
  __device__ explicit sink(char* o) : out(o) { }
  __device__ __forceinline__ char* at() { return W ? out + n : tmp; }
  __device__ __forceinline__ void ch(char c) { if(W) out[n] = c; ++n; }
  __device__ __forceinline__ void bytes(const char* s, uint64_t k) { if(W) for(uint64_t i = 0; i < k; ++i) out[n + i] = s[i]; n += (uint32_t)k; }
  __device__ __forceinline__ void i64(int64_t v) { n += mrfmt::fmt_int(at(), v); }
  __device__ __forceinline__ void u64(uint64_t v) { n += mrfmt::fmt_uint(at(), v); }
  __device__ __forceinline__ void g(double v) { n += mrfmt::fmt_general(at(), v); }
};

// ">N name\n" (compact format), for a read with rows or, with -0, without
template<bool W> __device__ uint32_t header(const crd_args& A, uint32_t r, char* out) {
  const uint64_t nrows = A.R.read_coords[r + 1] - A.R.read_coords[r];
  if(!A.compact || (nrows == 0 && !A.zero_match)) return 0;
  sink<W> s(out);
  s.ch('>'); s.u64(nrows); s.ch(' ');
  s.bytes(A.names + A.name_off[r], A.name_off[r + 1] - A.name_off[r]);
  s.ch('\n');
  return s.n;
}

// "[name ]%d %d %d %d %d %u %u %u %u %llu %u %g %g %g <super-read>[ %d:%d]...\n"
template<bool W> __device__ uint32_t row_line(const crd_args& A, uint64_t row, uint32_t r, char* out) {
  const coords_soa& c = A.R.c;
  sink<W> s(out);
  if(!A.compact) { s.bytes(A.names + A.name_off[r], A.name_off[r + 1] - A.name_off[r]); s.ch(' '); }
  s.i64(c.rs[row]); s.ch(' '); s.i64(c.re[row]); s.ch(' ');
  s.i64(c.qs[row]); s.ch(' '); s.i64(c.qe[row]); s.ch(' ');
  s.i64(c.nb_mers[row]); s.ch(' ');
  s.u64(c.pb_cons[row]); s.ch(' '); s.u64(c.sr_cons[row]); s.ch(' ');
  s.u64(c.pb_cover[row]); s.ch(' '); s.u64(c.sr_cover[row]); s.ch(' ');
  s.u64(A.R.read_len[r]); s.ch(' '); s.u64(c.ql[row]); s.ch(' ');
  s.g(c.stretch[row]); s.ch(' '); s.g(c.offset[row]); s.ch(' '); s.g(c.avg_err[row]); s.ch(' ');
  // super_reads::row_name: the header as read, or for a backward row with a path that path reversed and flipped
  const uint32_t sr = c.sr[row];
  const uint64_t pb = A.path_off[sr], pe = A.path_off[sr + 1];
  if(!c.use_bwd[row] || pb == pe) s.bytes(A.sr_names + A.sr_name_off[sr], A.sr_name_off[sr + 1] - A.sr_name_off[sr]);
  else
    for(uint64_t t = pe; t-- > pb;) {
      const uint32_t x = A.path_ids[t] ^ 1u;
      if(t + 1 < pe) s.ch('_');
      s.u64(x >> 1);
      s.ch((x & 1) ? 'R' : 'F');
    }
  const int32_t* ki = A.R.kinfo + c.info_off[row];
  const int32_t* bi = A.R.binfo + c.info_off[row];
  for(uint32_t t = 0; t < c.info_len[row]; ++t) { s.ch(' '); s.i64(ki[t]); s.ch(':'); s.i64(bi[t]); }
  s.ch('\n');
  return s.n;
}

__global__ void coords_measure_kernel(crd_args A) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t S = A.R.nrows;
  if(t < S) {
    const uint32_t r = A.R.c.read[t];
    uint32_t n = 0;
    if(A.R.c.sr[t] >= A.nseq) atomicMin(A.err, (unsigned long long)t);
    else n = row_line<false>(A, t, r, nullptr);
    A.len[t + r + 1] = n;
  } else if(t < S + A.R.nreads) {
    const uint32_t r = (uint32_t)(t - S);
    A.len[A.R.read_coords[r] + r] = header<false>(A, r, nullptr);
  }
}

__global__ void coords_emit_kernel(crd_args A) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t S = A.R.nrows;
  if(t < S) {
    const uint32_t r = A.R.c.read[t];
    row_line<true>(A, t, r, A.text + A.off[t + r + 1]);
  } else if(t < S + A.R.nreads) {
    const uint32_t r = (uint32_t)(t - S);
    header<true>(A, r, A.text + A.off[A.R.read_coords[r] + r]);
  }
}

} // namespace

extern "C" {

int mr_sr_names_create(mr_context* ctx, const char* names, const uint64_t* name_off, const uint32_t* path_ids,
                       const uint64_t* path_off, uint32_t nseq, mr_sr_names** out) {
  if(!ctx) return MR_EINVAL;
  if(!names || !name_off || !path_off || !out) return ctx->fail(MR_EINVAL, "mr_sr_names_create: null argument");
  *out = nullptr;
  if(!path_ids && path_off[nseq] != path_off[0]) return ctx->fail(MR_EINVAL, "mr_sr_names_create: null argument");
  for(uint32_t i = 0; i < nseq; ++i)
    if(name_off[i + 1] < name_off[i] || path_off[i + 1] < path_off[i])
      return ctx->fail(MR_EINVAL, "mr_sr_names_create: offsets must be non-decreasing");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  std::unique_ptr<mr_sr_names> s(new mr_sr_names);
  s->device = ctx->device; s->nseq = nseq;
  const uint64_t nbytes = name_off[nseq] - name_off[0], nids = path_off[nseq] - path_off[0];
  MR_TRY(s->names.ensure(ctx, nbytes + 1)); MR_TRY(s->name_off.ensure(ctx, ((size_t)nseq + 1) * 8));
  MR_TRY(s->path_ids.ensure(ctx, (nids + 1) * 4)); MR_TRY(s->path_off.ensure(ctx, ((size_t)nseq + 1) * 8));
  std::vector<uint64_t> rel(name_off, name_off + nseq + 1);
  for(auto& x : rel) x -= name_off[0];
  if(nbytes) MR_CUDA(ctx, cudaMemcpy(s->names.p, names + name_off[0], nbytes, cudaMemcpyHostToDevice));
  MR_CUDA(ctx, cudaMemcpy(s->name_off.p, rel.data(), rel.size() * 8, cudaMemcpyHostToDevice));
  rel.assign(path_off, path_off + nseq + 1);
  for(auto& x : rel) x -= path_off[0];
  if(nids) MR_CUDA(ctx, cudaMemcpy(s->path_ids.p, path_ids + path_off[0], nids * 4, cudaMemcpyHostToDevice));
  MR_CUDA(ctx, cudaMemcpy(s->path_off.p, rel.data(), rel.size() * 8, cudaMemcpyHostToDevice));
  *out = s.release();
  return MR_OK;
}

void mr_sr_names_destroy(mr_sr_names* s) {
  if(!s) return;
  cudaSetDevice(s->device);
  delete s;
}

int mr_coords_records(mr_context* ctx, const mr_result* res, const mr_coords_params* p, const mr_sr_names* srn,
                      const char* names, const uint64_t* name_off, mr_text** out) {
  if(!ctx) return MR_EINVAL;
  if(!res || !p || !srn || !names || !name_off || !out) return ctx->fail(MR_EINVAL, "mr_coords_records: null argument");
  *out = nullptr;
  mr_workspace* wsp = ctx->ws;
  if(res->ctx != ctx || !wsp || res->stamp == 0 || res->stamp != wsp->rows_stamp)
    return ctx->fail(MR_EINVAL, "mr_coords_records: the result is not the latest result of this context");
  if(srn->device != ctx->device) return ctx->fail(MR_EINVAL, "mr_coords_records: the super-read names live on another device");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  mr_workspace& ws = *wsp;
  cudaStream_t st = ctx->stream;
  std::unique_ptr<mr_text> t(new mr_text);
  t->ctx = ctx;
  const uint32_t nreads = ws.last_coords.nreads;
  if(nreads == 0) { *out = t.release(); return MR_OK; }

  crd_args A;
  memset(&A, 0, sizeof A);
  A.R = ws.last_coords;
  A.sr_names = srn->names.as<char>(); A.sr_name_off = srn->name_off.as<uint64_t>();
  A.path_ids = srn->path_ids.as<uint32_t>(); A.path_off = srn->path_off.as<uint64_t>(); A.nseq = srn->nseq;
  A.compact = p->compact != 0; A.zero_match = p->zero_match != 0;
  const uint64_t nslots = A.R.nrows + nreads;
  // per slot its length and its offset, then the error word and the total
  MR_TRY(ws.rec_lines.ensure(ctx, nslots * 12 + 64));
  { char* q = ws.rec_lines.as<char>(); A.off = (const uint64_t*)q; A.len = (uint32_t*)(q + nslots * 8);
    A.err = (unsigned long long*)(((uintptr_t)(q + nslots * 12) + 15) & ~(uintptr_t)15); }
  uint64_t* d_total = (uint64_t*)A.err + 1;
  MR_TRY(upload_read_names(ctx, ws, names, name_off, nreads, &A.name_off, &A.names));
  MR_CUDA(ctx, cudaMemsetAsync(A.err, 0xff, 8, st));
  coords_measure_kernel<<<div_up(nslots, 256), 256, 0, st>>>(A);
  MR_LAUNCHED(ctx);
  MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ A.len }, nslots, (uint64_t*)A.off, ws.scan_scratch, d_total)));
  uint64_t h[2] = { ~0ULL, 0 };
  MR_CUDA(ctx, cudaMemcpyAsync(h, A.err, 16, cudaMemcpyDeviceToHost, st));
  MR_CUDA(ctx, ctx->wait(st));
  if(h[0] != ~0ULL)
    return ctx->fail(MR_EINVAL, "mr_coords_records: row " + std::to_string(h[0]) + " refers to a super-read that the names do not have (" +
                                std::to_string(srn->nseq) + " super-reads)");
  const uint64_t bytes = h[1];
  MR_TRY(take_text_slab(ctx, ws, t.get(), bytes));
  if(bytes) {
    MR_TRY(ws.rec_text.ensure(ctx, bytes + 1));
    A.text = ws.rec_text.as<char>();
    coords_emit_kernel<<<div_up(nslots, 256), 256, 0, st>>>(A);
    MR_LAUNCHED(ctx);
    MR_CUDA(ctx, cudaMemcpyAsync(t->host->p, A.text, bytes, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
  }
  *out = t.release();
  return MR_OK;
}

} // extern "C"

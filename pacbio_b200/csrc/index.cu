// Suffix-array construction and batched k-mer lookup on the device.
// Replaces the reference's PSA::PSA -> SA::create_mt (psa.hpp:130-140, mer_sa_imp.hpp:197-267:
// histogram, partial sums, atomic scatter, 4^m std::sort calls) by one stable LSD radix sort of
// (padded k-mer, position) pairs seeded in descending position order, and PSA::search
// (mer_sa_imp.hpp:369-479) by a prefix-table probe plus a scan of the bucket's tails.
#include <cstdio>
#include <cstdlib>
#include "index.cuh"
#include "primitives.cuh"

#include <algorithm>
#include <cstring>
#include <memory>

int build_slots(mr_index* idx);

namespace {

// k-mer starting at `pos`, first base most significant, bases past the end of the text read as A
__device__ __forceinline__ uint64_t text_kmer(const uint64_t* __restrict__ text, uint64_t pos, uint32_t k) {
  const uint64_t w = pos >> 5;
  const unsigned sh = (unsigned)(pos & 31) * 2;
  const uint64_t w0 = text[w], w1 = text[w + 1];
  const uint64_t raw = sh ? ((w0 >> sh) | (w1 << (64 - sh))) : w0;
  return reverse_pairs(raw) >> (64 - 2 * k);
}

__global__ void clear_text_tail_kernel(uint64_t* text, uint64_t n) {
  const uint64_t w = n >> 5;
  const unsigned used = (unsigned)(n & 31) * 2;
  if(used) text[w] &= (1ULL << used) - 1; else text[w] = 0;
  text[w + 1] = 0;
}

// entry i holds position nsa-1-i: the stable sort then leaves equal k-mers in descending position
__global__ void __launch_bounds__(256) sa_keys_kernel(const uint64_t* __restrict__ text, uint32_t nsa, uint32_t k,
                                                      uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nsa; i += stride) {
    const uint32_t pos = nsa - 1 - i;
    keys[i] = text_kmer(text, pos, k);
    vals[i] = pos;
  }
}

// tails + prefix counts from the sorted keys: counts[v] = first rank whose m-mer is >= v.
// Runs of empty prefixes longer than kGapInline are queued and filled by whole CTAs afterwards
// (a tiny text leaves almost all of the 4^m prefixes empty).
constexpr int kGapInline = 256;
struct gap_item { uint32_t first, last, value; };

template<typename TailT>
__global__ void __launch_bounds__(256) sa_finish_kernel(const uint64_t* __restrict__ keys, uint32_t nsa, uint32_t tail_bits,
                                                        uint32_t nprefix, TailT* __restrict__ tails,
                                                        uint32_t* __restrict__ counts,
                                                        gap_item* __restrict__ gaps, uint32_t* __restrict__ ngaps) {
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint64_t tmask = tail_bits >= 64 ? ~0ULL : ((1ULL << tail_bits) - 1);
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= nsa; i += stride) {
    // i == nsa is the virtual end: fills counts above the last occupied prefix
    const int64_t prev = i == 0 ? -1 : (int64_t)(keys[i - 1] >> tail_bits);
    const int64_t cur  = i == nsa ? (int64_t)nprefix : (int64_t)(keys[i] >> tail_bits);
    if(i < nsa && tails) tails[i] = (TailT)(keys[i] & tmask);
    if(cur - prev <= kGapInline) {
      for(int64_t v = prev + 1; v <= cur; ++v) counts[v] = i;
    } else {
      const uint32_t slot = atomicAdd(ngaps, 1u);
      gaps[slot] = gap_item{ (uint32_t)(prev + 1), (uint32_t)cur, i };
    }
  }
}

// keys of the sorted entries recomputed from the text (for the parity tap that exports the
// reference's 4^psa_min + 1 table)
__global__ void __launch_bounds__(256) sa_rekey_kernel(const uint64_t* __restrict__ text, const uint32_t* __restrict__ sa,
                                                       uint32_t nsa, uint32_t k, uint64_t* __restrict__ keys) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nsa; i += stride) keys[i] = text_kmer(text, sa[i], k);
}

__global__ void __launch_bounds__(256) sa_fill_gaps_kernel(const gap_item* __restrict__ gaps, const uint32_t* __restrict__ ngaps,
                                                           uint32_t* __restrict__ counts) {
  const uint32_t n = *ngaps;
  for(uint32_t g = blockIdx.x; g < n; g += gridDim.x) {
    const gap_item it = gaps[g];
    for(uint64_t v = (uint64_t)it.first + threadIdx.x; v <= it.last; v += blockDim.x) counts[v] = it.value;
  }
}

__global__ void __launch_bounds__(256) blk_table_kernel(const uint32_t* __restrict__ sr_start, uint32_t nseq,
                                                        uint32_t nblk, uint32_t* __restrict__ blk) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if(b >= nblk) return;
  const uint64_t x = (uint64_t)b << kBlkShift;
  uint32_t lo = 0, hi = nseq;                 // largest i in [0, nseq) with sr_start[i] <= x
  while(hi - lo > 1) { const uint32_t mid = lo + ((hi - lo) >> 1); if(sr_start[mid] <= x) lo = mid; else hi = mid; }
  blk[b] = lo;
}

__global__ void __launch_bounds__(256) blkx_kernel(const uint32_t* __restrict__ blk, const uint32_t* __restrict__ sr_start, uint32_t nblk,
                                                   uint4* __restrict__ blkx) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if(b >= nblk) return;
  const uint32_t i = blk[b];
  blkx[b] = make_uint4(i, sr_start[i], sr_start[i + 1], 0u);
}

__global__ void __launch_bounds__(256) widen_kernel(const uint32_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ out) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = in[i];
}

// one thread per query.  Every query makes two dependent, effectively random HBM accesses
// (8 bytes of the prefix table, then the bucket's tails): the kernel is bound by random-sector
// throughput, so all it needs is enough independent loads in flight per SM.
__global__ void __launch_bounds__(256) lookup_kernel(index_view iv, const uint64_t* __restrict__ mers, uint64_t q,
                                                     uint64_t* __restrict__ index_out, uint64_t* __restrict__ nb_out) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < q; i += stride) {
    uint32_t idx, nb;
    index_lookup(iv, mers[i], idx, nb);
    index_out[i] = idx;
    nb_out[i]    = nb;
  }
}

// located suffix-array entries (index_view::saloc)
__global__ void __launch_bounds__(256) saloc_kernel(index_view iv, uint2* __restrict__ saloc) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < iv.nsa; i += stride) {
    uint32_t sr, off;
    const uint32_t x = iv.sa[i];
    // (positions of a part's extension belong to the next part and never match here: index.cuh)
    saloc[i] = x < iv.own && index_locate(iv, x, sr, off) ? make_uint2(sr, off) : make_uint2(0xffffffffu, 0u);
  }
}

// nibble records (index_view::nib): one thread per group of 32 prefixes
__global__ void __launch_bounds__(256) nib_kernel(const uint32_t* __restrict__ counts, uint32_t ngroups, ulonglong2* __restrict__ nib,
                                                  uint32_t* __restrict__ gbase, unsigned long long* __restrict__ n_overflow) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if(g >= ngroups) return;
  const uint32_t* c = counts + (uint64_t)g * 32;
  uint64_t w[2] = { 0, 0 };
  bool big = false;
  uint32_t prev = c[0];
  for(int j = 0; j < 32; ++j) {
    const uint32_t next = c[j + 1], sz = next - prev;
    prev = next;
    big |= sz >= 15;
    w[j >> 4] |= (uint64_t)(sz & 15u) << (4 * (j & 15));
  }
  if(big) { w[0] |= 15ULL; atomicAdd(n_overflow, 1ULL); }    // marker: this group is looked up in counts[]
  nib[g] = make_ulonglong2(w[0], w[1]);
  gbase[g] = c[0];
}

// random-sector ceiling: every thread issues 8 independent 16-byte loads per round at hashed places
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
__global__ void __launch_bounds__(256) random_gather_kernel(const uint4* __restrict__ table, uint64_t nelem, uint32_t rounds,
                                                            uint32_t salt, uint32_t* __restrict__ sink) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t acc = 0;
  for(uint32_t r = 0; r < rounds; ++r) {
    uint4 v[8];
#pragma unroll
    for(int j = 0; j < 8; ++j) {
      const uint64_t h = ((uint64_t)mix32((tid * 8u + j + salt) ^ mix32(r + 0x9e3779b9u)) << 32) | mix32((r + 1) * 0x9e3779b9u ^ (tid + j * 0x85ebca6bu));
      v[j] = __ldg(table + (uint64_t)(((unsigned __int128)h * nelem) >> 64));
    }
#pragma unroll
    for(int j = 0; j < 8; ++j) acc ^= v[j].x ^ v[j].y ^ v[j].z ^ v[j].w;
  }
  if(acc == 0x12345678u) sink[0] = acc;          // keeps the loads alive
}

} // namespace

// prefix table over `mp` bases (and, when tails != null, the tails) from the sorted keys
static int build_prefix_table(mr_context* ctx, const uint64_t* keys, uint32_t nsa, uint32_t k, uint32_t mp,
                              void* tails, uint32_t tail_bytes, uint32_t* counts) {
  cudaStream_t st = ctx->stream;
  const uint32_t tail_bits = 2 * (k - mp);
  const uint32_t nprefix = 1u << (2 * mp);
  dev_buf gaps;
  const uint32_t max_gaps = nprefix / kGapInline + 2;
  MR_TRY(gaps.ensure(ctx, (size_t)max_gaps * sizeof(gap_item) + 16));
  uint32_t* ngaps = reinterpret_cast<uint32_t*>(gaps.as<gap_item>() + max_gaps);
  MR_CUDA(ctx, cudaMemsetAsync(ngaps, 0, sizeof(uint32_t), st));
  const unsigned grid = ctx->sm_count * 8;
  if(tail_bytes == 1) sa_finish_kernel<uint8_t><<<grid, 256, 0, st>>>(keys, nsa, tail_bits, nprefix, (uint8_t*)tails, counts, gaps.as<gap_item>(), ngaps);
  else if(tail_bytes == 2) sa_finish_kernel<uint16_t><<<grid, 256, 0, st>>>(keys, nsa, tail_bits, nprefix, (uint16_t*)tails, counts, gaps.as<gap_item>(), ngaps);
  else sa_finish_kernel<uint32_t><<<grid, 256, 0, st>>>(keys, nsa, tail_bits, nprefix, (uint32_t*)tails, counts, gaps.as<gap_item>(), ngaps);
  MR_LAUNCHED(ctx);
  sa_fill_gaps_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(gaps.as<gap_item>(), ngaps, counts);
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaStreamSynchronize(st));       // gaps is a local buffer
  return MR_OK;
}

// Internal prefix length: as long as psa_min allows, small enough that prefix table + tails stay
// L2 resident (budget 110 MB of the 126 MB), but never so small that the mean bucket exceeds ~32.
static uint32_t choose_internal_prefix(uint64_t n, uint32_t psa_min, uint32_t k) {
  uint32_t lo = 1;
  while(lo < psa_min && ((uint64_t)1 << (2 * lo)) * 32 < n) ++lo;            // mean bucket <= 32
  uint32_t best = psa_min;
  while(best > lo) {
    const uint32_t tb = 2 * (k - best);
    const uint64_t bytes = (((uint64_t)1 << (2 * best)) + 1) * 4 + n * (tb <= 8 ? 1 : (tb <= 16 ? 2 : 4));
    if(bytes <= (110ULL << 20)) break;
    --best;
  }
  if(const char* e = getenv("MR_INDEX_PREFIX")) {           // tuning knob: force the internal prefix length
    const uint32_t v = (uint32_t)atoi(e);
    if(v >= 1 && v < k && v <= 15) best = v;                // (it may exceed --psa-min: buckets are cut from the fully sorted keys)
  }
  while(k - best > (uint32_t)kMaxShort) ++best;
  return best;
}

// One part: a complete index over `n` bases of text.  sr_start[0 .. nseq] are the part's own
// super-read starts (sr_start[nseq] = its own bases <= n; the rest of the text, if any, is the
// extension described in index.cuh).
static int build_part(mr_context* ctx, const uint64_t* text2bit, uint64_t n, const uint64_t* sr_start, uint32_t nseq,
                      uint32_t psa_min, uint32_t k, mr_index** out) {
  if(n > 0xff000000ULL + 64) return ctx->fail(MR_ELIMIT, "mr_index_create: index part of 2^32 bases or more");
  phase_timer timer(ctx);

  std::unique_ptr<mr_index> idx(new mr_index);
  idx->ctx = ctx; idx->n = n; idx->k = k; idx->m = psa_min; idx->nseq = nseq;
  idx->nsa = (uint32_t)(n - psa_min + 1);
  const uint32_t nsa = idx->nsa;
  const uint64_t nwords = (n + 31) / 32;
  const uint32_t mi = choose_internal_prefix(n, psa_min, k);
  idx->mi = mi;
  const uint32_t tail_bits = 2 * (k - mi);
  const uint32_t tail_bytes = tail_bits <= 8 ? 1 : (tail_bits <= 16 ? 2 : 4);
  const uint32_t nprefix = 1u << (2 * mi);
  cudaStream_t st = ctx->stream;

  timer.begin("Super read upload");
  MR_TRY(idx->text.ensure(ctx, (nwords + 2) * sizeof(uint64_t)));
  MR_CUDA(ctx, cudaMemsetAsync(idx->text.as<uint64_t>() + nwords, 0, 2 * sizeof(uint64_t), st));
  MR_CUDA(ctx, cudaMemcpyAsync(idx->text.p, text2bit, nwords * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  clear_text_tail_kernel<<<1, 1, 0, st>>>(idx->text.as<uint64_t>(), n);
  MR_LAUNCHED(ctx);
  {
    std::vector<uint32_t> starts32(nseq + 1);
    for(uint32_t i = 0; i <= nseq; ++i) starts32[i] = (uint32_t)sr_start[i];
    MR_TRY(idx->sr_start.ensure(ctx, ((size_t)nseq + 2) * sizeof(uint32_t)));
    MR_CUDA(ctx, cudaMemcpyAsync(idx->sr_start.p, starts32.data(), ((size_t)nseq + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  const uint32_t nblk = (uint32_t)(n >> kBlkShift) + 1;
  MR_TRY(idx->blk.ensure(ctx, ((size_t)nblk + 1) * sizeof(uint32_t)));
  blk_table_kernel<<<div_up(nblk, 256), 256, 0, st>>>(idx->sr_start.as<uint32_t>(), nseq, nblk, idx->blk.as<uint32_t>());
  MR_LAUNCHED(ctx);

  timer.next("sorting");
  {
    dev_buf k0, k1, v0, v1;
    prim::sort_scratch scratch;
    MR_TRY(k0.ensure(ctx, (size_t)nsa * sizeof(uint64_t)));
    MR_TRY(k1.ensure(ctx, (size_t)nsa * sizeof(uint64_t)));
    MR_TRY(v0.ensure(ctx, (size_t)nsa * sizeof(uint32_t)));
    MR_TRY(v1.ensure(ctx, (size_t)nsa * sizeof(uint32_t)));
    sa_keys_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(idx->text.as<uint64_t>(), nsa, k, k0.as<uint64_t>(), v0.as<uint32_t>());
    MR_LAUNCHED(ctx);
    bool in_first = true;
    MR_TRY((prim::radix_sort_pairs<uint64_t, uint32_t>(ctx, k0.as<uint64_t>(), v0.as<uint32_t>(), k1.as<uint64_t>(),
                                                       v1.as<uint32_t>(), nsa, 0, 2 * (int)k, scratch, &in_first)));
    timer.next("partial sums");
    const uint64_t* keys = in_first ? k0.as<uint64_t>() : k1.as<uint64_t>();
    dev_buf& vres = in_first ? v0 : v1;
    MR_TRY(idx->alloc_lut(ctx, ((size_t)nprefix + 8) * sizeof(uint32_t),       // counts are read in 16-byte blocks
                          ((size_t)nsa + 64) * tail_bytes));
    MR_TRY(build_prefix_table(ctx, keys, nsa, k, mi, idx->tails.p, tail_bytes, idx->counts.as<uint32_t>()));
    // keep the sorted positions: steal the buffer that holds them
    MR_CUDA(ctx, cudaStreamSynchronize(st));
    std::swap(idx->sa.p, vres.p);
    std::swap(idx->sa.cap, vres.cap);
  }
  timer.end();
  MR_CUDA(ctx, cudaStreamSynchronize(st));
  timer.collect();

  // tail-short suffixes: positions n-k+1 .. n-m, padded k-mers computed on the host from the 2-bit text
  index_view& v = idx->view;
  v.counts = idx->counts.as<uint32_t>(); v.tails = idx->tails.p; v.sa = idx->sa.as<uint32_t>();
  v.sr_start = idx->sr_start.as<uint32_t>(); v.blk = idx->blk.as<uint32_t>();
  v.n = n; v.nsa = nsa; v.nseq = nseq; v.k = k; v.m = psa_min; v.mi = mi; v.tail_bits = tail_bits; v.tail_bytes = tail_bytes;
  v.sr_base = 0; v.nseq_all = nseq; v.own = (uint32_t)sr_start[nseq];
  MR_TRY(build_slots(idx.get()));
  v.nshort = 0;
  for(uint32_t j = 1; j <= k - psa_min; ++j) {
    const uint64_t pos = n - k + j;
    uint64_t key = 0;
    for(uint32_t t = 0; t < k; ++t) {
      const uint64_t p = pos + t;
      const uint64_t c = p < n ? (text2bit[p >> 5] >> (2 * (p & 31))) & 3 : 0;
      key = (key << 2) | c;
    }
    v.short_key[v.nshort++] = key;
  }
  idx->n_all = sr_start[nseq]; idx->nseq_all = nseq;
  *out = idx.release();
  return MR_OK;
}

// derived tables of a part whose arrays are in place (after a build or a load): blkx, and the slot table
int build_slots(mr_index* idx) {
  mr_context* ctx = idx->ctx;
  index_view& v = idx->view;
  {
    const uint32_t nblk = (uint32_t)(idx->n >> kBlkShift) + 1;
    MR_TRY(idx->blkx.ensure(ctx, (size_t)nblk * sizeof(uint4)));
    blkx_kernel<<<div_up(nblk, 256), 256, 0, ctx->stream>>>(idx->blk.as<uint32_t>(), idx->sr_start.as<uint32_t>(), nblk, idx->blkx.as<uint4>());
    MR_LAUNCHED(ctx);
    MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    v.blkx = idx->blkx.as<uint4>();
  }
  v.saloc = nullptr;
  MR_TRY(idx->saloc.ensure(ctx, (size_t)v.nsa * sizeof(uint2)));
  saloc_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(v, idx->saloc.as<uint2>());
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  v.saloc = idx->saloc.as<uint2>();
  v.nib = nullptr; v.gbase = nullptr;
  // The nibble form of the prefix counts pays while most groups of 64 buckets hold no bucket of 15 entries:
  // a mean bucket of up to ~4 (the yeast-size index: 2.1).
  const uint32_t nprefix = 1u << (2 * v.mi);
  if(v.mi < 3 || (uint64_t)v.nsa > (uint64_t)nprefix * 4) return MR_OK;
  const uint32_t ngroups = nprefix / 32;
  MR_TRY(idx->nib.ensure(ctx, (size_t)ngroups * sizeof(ulonglong2)));
  MR_TRY(idx->gbase.ensure(ctx, (size_t)ngroups * sizeof(uint32_t)));
  dev_buf ovf;
  MR_TRY(ovf.ensure(ctx, sizeof(unsigned long long)));
  MR_CUDA(ctx, cudaMemsetAsync(ovf.p, 0, sizeof(unsigned long long), ctx->stream));
  nib_kernel<<<div_up(ngroups, 256), 256, 0, ctx->stream>>>(idx->counts.as<uint32_t>(), ngroups, idx->nib.as<ulonglong2>(), idx->gbase.as<uint32_t>(),
                                                          ovf.as<unsigned long long>());
  MR_LAUNCHED(ctx);
  unsigned long long n_overflow = 0;
  MR_CUDA(ctx, cudaMemcpyAsync(&n_overflow, ovf.p, sizeof n_overflow, cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if(n_overflow * 4 > ngroups) { idx->nib.release(); idx->gbase.release(); return MR_OK; }    // too many groups fall back: not worth the extra read
  v.nib = idx->nib.as<ulonglong2>(); v.gbase = idx->gbase.as<uint32_t>();
  idx->nib_overflow_groups = n_overflow;
  return MR_OK;
}

// whole-index tables of a freshly built or loaded one-part index: the super-read lengths
int finish_single_part(mr_index* idx, const std::vector<uint32_t>& sr_len) {
  mr_context* ctx = idx->ctx;
  MR_TRY(idx->sr_len.ensure(ctx, (sr_len.size() + 1) * sizeof(uint32_t)));
  MR_CUDA(ctx, cudaMemcpyAsync(idx->sr_len.p, sr_len.data(), sr_len.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

// bases [from, from + len) of a 2-bit text as a text of its own (base 0 at bit 0 of word 0)
static void slice_text(const uint64_t* text, uint64_t from, uint64_t len, std::vector<uint64_t>& out) {
  const uint64_t nwords = (len + 31) / 32, last = (from + len - 1) >> 5;
  out.assign(nwords + 2, 0);
  const uint64_t w0 = from >> 5;
  const unsigned sh = (unsigned)(from & 31) * 2;
  for(uint64_t i = 0; i < nwords; ++i) {
    const uint64_t lo = text[w0 + i];
    const uint64_t hi = (sh && w0 + i + 1 <= last) ? text[w0 + i + 1] : 0;
    out[i] = sh ? ((lo >> sh) | (hi << (64 - sh))) : lo;
  }
  if(len & 31) out[nwords - 1] &= (1ULL << (2 * (len & 31))) - 1;
}

extern "C" {

int mr_index_create(mr_context* ctx, const uint64_t* text2bit, uint64_t n, const uint64_t* sr_start, uint32_t nseq,
                    const uint32_t* unitig_ids, const uint64_t* unitig_off, const int32_t* unitig_len,
                    uint32_t n_unitigs, uint32_t psa_min, uint32_t k, mr_index** out) {
  if(!ctx) return MR_EINVAL;
  if(!out || !text2bit || !sr_start || nseq == 0) return ctx->fail(MR_EINVAL, "mr_index_create: null argument");
  if(!(psa_min >= 1 && psa_min < k && k <= 31))
    return ctx->fail(MR_EINVAL, "mr_index_create: need 1 <= psa_min < mer <= 31");
  if(psa_min > 15) return ctx->fail(MR_ELIMIT, "mr_index_create: psa_min > 15 (prefix table over 4 GiB) not supported");
  if(k - psa_min > (uint32_t)kMaxShort) return ctx->fail(MR_ELIMIT, "mr_index_create: mer - psa_min > 16 not supported");
  if(n < k) return ctx->fail(MR_EINVAL, "mr_index_create: text shorter than one k-mer");
  if(sr_start[0] != 0 || sr_start[nseq] != n) return ctx->fail(MR_EINVAL, "mr_index_create: sr_start must span [0, n]");
  if(nseq >= 0xfffffff0u) return ctx->fail(MR_ELIMIT, "mr_index_create: 2^32 super-reads or more not supported");
  std::vector<uint32_t> sr_len(nseq);
  for(uint32_t i = 0; i < nseq; ++i) {
    if(sr_start[i + 1] <= sr_start[i]) return ctx->fail(MR_EINVAL, "mr_index_create: sr_start must be strictly increasing");
    if(sr_start[i + 1] - sr_start[i] >= (1ULL << 31)) return ctx->fail(MR_ELIMIT, "mr_index_create: super-read of 2^31 bases or more");
    sr_len[i] = (uint32_t)(sr_start[i + 1] - sr_start[i]);
  }
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->timers.clear();
  cudaStream_t st = ctx->stream;

  // ---- parts (index.cuh): one unless the text has 2^32 bases or more ------------------------------
  // MR_INDEX_PART_BASES lowers the limit (the tests force several parts on small inputs)
  // 2^32 - 2^24: grid-stride loops over 32-bit ranks must not wrap
  uint64_t part_limit = 0xff000000ULL;
  if(const char* e = getenv("MR_INDEX_PART_BASES")) { const uint64_t v = strtoull(e, nullptr, 0); if(v >= 1024 && v < part_limit) part_limit = v; }
  const uint64_t ext_max = k - 1;
  std::vector<uint32_t> cut;            // part p = super-reads [cut[p], cut[p + 1])
  cut.push_back(0);
  if(n + 0 > part_limit) {
    const uint64_t nparts = (n + part_limit - ext_max - 1) / (part_limit - ext_max);
    if(nparts > (uint64_t)kMaxParts) return ctx->fail(MR_ELIMIT, "mr_index_create: text too long (more than 4 index parts)");
    for(uint64_t p = 1; p < nparts; ++p) {
      const uint64_t target = n / nparts * p;
      uint32_t i = (uint32_t)(std::lower_bound(sr_start, sr_start + nseq, target) - sr_start);
      if(i <= cut.back()) i = cut.back() + 1;
      if(i >= nseq) break;
      cut.push_back(i);
    }
  }
  cut.push_back(nseq);
  const uint32_t P = (uint32_t)cut.size() - 1;

  std::unique_ptr<mr_index> idx;
  for(uint32_t p = 0; p < P; ++p) {
    const uint64_t from = sr_start[cut[p]], own = sr_start[cut[p + 1]] - from;
    const uint64_t ext = std::min<uint64_t>(ext_max, n - (from + own));
    if(own + ext > 0xff000000ULL + 64)
      return ctx->fail(MR_ELIMIT, "mr_index_create: cannot cut the super-reads into parts of fewer than 2^32 bases");
    const uint32_t pseq = cut[p + 1] - cut[p];
    mr_index* part = nullptr;
    if(P == 1) {
      MR_TRY(build_part(ctx, text2bit, n, sr_start, nseq, psa_min, k, &part));
    } else {
      std::vector<uint64_t> ptext, pstart(pseq + 1);
      slice_text(text2bit, from, own + ext, ptext);
      for(uint32_t i = 0; i <= pseq; ++i) pstart[i] = sr_start[cut[p] + i] - from;
      MR_TRY(build_part(ctx, ptext.data(), own + ext, pstart.data(), pseq, psa_min, k, &part));
    }
    part->view.sr_base = cut[p];
    part->view.nseq_all = nseq;
    if(p == 0) idx.reset(part); else idx->more.push_back(part);
  }
  idx->n_all = n; idx->nseq_all = nseq;
  if(getenv("MR_TRACE") || (P > 1 && getenv("MR_SHOW_TIMING"))) {
    fprintf(stderr, "[mr] index parts: %u (", P);
    for(uint32_t p = 0; p < P; ++p) fprintf(stderr, "%s%llu", p ? " + " : "", (unsigned long long)(sr_start[cut[p + 1]] - sr_start[cut[p]]));
    fprintf(stderr, " bases)\n");
  }
  MR_TRY(finish_single_part(idx.get(), sr_len));
  if(P > 1) {
    std::vector<index_view> views(P - 1);
    for(uint32_t p = 1; p < P; ++p) views[p - 1] = idx->more[p - 1]->view;
    MR_TRY(idx->more_views.ensure(ctx, views.size() * sizeof(index_view)));
    MR_CUDA(ctx, cudaMemcpyAsync(idx->more_views.p, views.data(), views.size() * sizeof(index_view), cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaStreamSynchronize(st));
  }

  if(unitig_ids && unitig_off && unitig_len && n_unitigs) {
    idx->has_unitigs = true;
    idx->n_unitigs = n_unitigs;
    const uint64_t total = unitig_off[nseq];
    idx->unitig_total = total;
    for(uint32_t i = 0; i < nseq; ++i)
      if(unitig_off[i + 1] < unitig_off[i]) return ctx->fail(MR_EINVAL, "mr_index_create: unitig_off must be non-decreasing");
    // A path may name a k-unitig the -l/-u table does not have (a stray super-read name): coords and
    // kmers_info handle that like the reference (pb_aligner.cc:103-143 clears the row's vectors), but the
    // overlap graph indexes the length table with these ids unchecked -- mr_align_batch refuses to run
    // it on such an index instead of reading out of bounds.
    uint32_t max_uid = 0;
    for(uint64_t i = 0; i < total; ++i) max_uid = std::max(max_uid, unitig_ids[i] >> 1);
    idx->unitig_ids_ok = total == 0 || max_uid < n_unitigs;
    MR_TRY(idx->unitig_ids.ensure(ctx, (total + 1) * sizeof(uint32_t)));
    MR_TRY(idx->unitig_off.ensure(ctx, ((size_t)nseq + 1) * sizeof(uint64_t)));
    MR_TRY(idx->unitig_len.ensure(ctx, (size_t)n_unitigs * sizeof(int32_t)));
    MR_CUDA(ctx, cudaMemcpyAsync(idx->unitig_ids.p, unitig_ids, total * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaMemcpyAsync(idx->unitig_off.p, unitig_off, ((size_t)nseq + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaMemcpyAsync(idx->unitig_len.p, unitig_len, (size_t)n_unitigs * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  idx->inputs_checksum = mr_inputs_checksum(text2bit, n, sr_start, nseq, unitig_ids, unitig_off, unitig_len, n_unitigs, psa_min, k);
  *out = idx.release();
  return MR_OK;
}

void mr_index_destroy(mr_index* idx) {
  if(!idx) return;
  cudaSetDevice(idx->ctx->device);
  delete idx;
}

uint64_t mr_index_sa_size(const mr_index* idx) { return idx ? idx->nsa : 0; }
uint32_t mr_index_parts(const mr_index* idx) { return idx ? idx->nparts() : 0; }
uint64_t mr_index_table_bytes(const mr_index* idx) {
  if(!idx) return 0;
  auto part_bytes = [](const mr_index* p) -> uint64_t {
    if(!p->view.nib) return p->lut_bytes;
    // with nibble records the prefix counts are only read for the groups that overflow
    const uint64_t ngroups = (1ULL << (2 * p->mi)) / 32;
    return ngroups * 20 + ((uint64_t)p->nsa + 64) * p->view.tail_bytes + p->nib_overflow_groups * 132;
  };
  uint64_t b = part_bytes(idx);
  for(const mr_index* p : idx->more) b += part_bytes(p);
  return b;
}

static int export_widened(mr_index* idx, const uint32_t* d_in, uint64_t count, uint64_t* h_out) {
  mr_context* ctx = idx->ctx;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  dev_buf tmp;
  MR_TRY(tmp.ensure(ctx, count * sizeof(uint64_t)));
  widen_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_in, count, tmp.as<uint64_t>());
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaMemcpyAsync(h_out, tmp.p, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

// The taps and PSA::search below speak in ranks of ONE suffix array: they are defined for a
// one-part index (every text below 2^32 bases).
#define MR_ONE_PART(idx, what) do { if((idx)->nparts() > 1) return (idx)->ctx->fail(MR_ELIMIT, what ": not defined for an index of several parts (text of 2^32 bases or more)"); } while(0)

int mr_index_export_sa(mr_index* idx, uint64_t* sa_out) {
  if(!idx || !sa_out) return MR_EINVAL;
  MR_ONE_PART(idx, "mr_index_export_sa");
  return export_widened(idx, idx->sa.as<uint32_t>(), idx->nsa, sa_out);
}

int mr_index_export_counts(mr_index* idx, uint64_t* counts_out) {
  if(!idx || !counts_out) return MR_EINVAL;
  MR_ONE_PART(idx, "mr_index_export_counts");
  mr_context* ctx = idx->ctx;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  // the reference's table is over psa_min bases; ours is over mi <= psa_min: rebuild it from the text
  dev_buf keys, counts;
  const uint32_t nprefix = 1u << (2 * idx->m);
  MR_TRY(keys.ensure(ctx, (size_t)idx->nsa * sizeof(uint64_t)));
  MR_TRY(counts.ensure(ctx, ((size_t)nprefix + 8) * sizeof(uint32_t)));
  sa_rekey_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(idx->text.as<uint64_t>(), idx->sa.as<uint32_t>(), idx->nsa, idx->k,
                                                             keys.as<uint64_t>());
  MR_LAUNCHED(ctx);
  MR_TRY(build_prefix_table(ctx, keys.as<uint64_t>(), idx->nsa, idx->k, idx->m, nullptr, 4, counts.as<uint32_t>()));
  dev_buf tmp;
  const uint64_t count = (uint64_t)nprefix + 1;
  MR_TRY(tmp.ensure(ctx, count * sizeof(uint64_t)));
  widen_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(counts.as<uint32_t>(), count, tmp.as<uint64_t>());
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaMemcpyAsync(counts_out, tmp.p, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

int mr_selftest_random_gather(mr_context* ctx, uint64_t table_bytes, uint64_t loads, double* sector_gbs) {
  if(!ctx) return MR_EINVAL;
  if(!sector_gbs || table_bytes < 4096 || loads == 0) return ctx->fail(MR_EINVAL, "mr_selftest_random_gather: bad argument");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  dev_buf table, sink;
  MR_TRY(table.ensure(ctx, table_bytes));
  MR_TRY(sink.ensure(ctx, 64));
  MR_CUDA(ctx, cudaMemsetAsync(table.p, 0x5a, table_bytes, ctx->stream));
  const unsigned grid = ctx->sm_count * 8;
  const uint64_t per_round = (uint64_t)grid * 256 * 8;
  const uint32_t rounds = (uint32_t)std::max<uint64_t>(1, (loads + per_round - 1) / per_round);
  cudaEvent_t a, b;
  MR_CUDA(ctx, cudaEventCreate(&a)); MR_CUDA(ctx, cudaEventCreate(&b));
  double best = 0.0;
  for(int rep = 0; rep < 4; ++rep) {              // the first launch warms up
    cudaEventRecord(a, ctx->stream);
    random_gather_kernel<<<grid, 256, 0, ctx->stream>>>(table.as<uint4>(), table_bytes / 16, rounds, 977u * rep, sink.as<uint32_t>());
    MR_LAUNCHED(ctx);
    cudaEventRecord(b, ctx->stream);
    cudaError_t e = cudaEventSynchronize(b);
    if(e != cudaSuccess) { cudaEventDestroy(a); cudaEventDestroy(b); return ctx->fail(MR_ECUDA, cudaGetErrorString(e)); }
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    if(rep && ms > 0) best = std::max(best, (double)rounds * per_round * 32.0 / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(a); cudaEventDestroy(b);
  *sector_gbs = best;
  return MR_OK;
}

int mr_lookup_batch_device(mr_index* idx, const uint64_t* d_mers, uint64_t q, uint64_t* d_index_out, uint64_t* d_nb_out) {
  if(!idx) return MR_EINVAL;
  MR_ONE_PART(idx, "mr_lookup_batch");
  mr_context* ctx = idx->ctx;
  if(q == 0) return MR_OK;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count * 8, div_up(q, 256));
  lookup_kernel<<<grid, 256, 0, ctx->stream>>>(idx->view, d_mers, q, d_index_out, d_nb_out);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

int mr_lookup_batch(mr_index* idx, const uint64_t* mers, uint64_t q, uint64_t* index_out, uint64_t* nb_out) {
  if(!idx || !mers || !index_out || !nb_out) return MR_EINVAL;
  mr_context* ctx = idx->ctx;
  if(q == 0) return MR_OK;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  dev_buf dm, di, dn;
  MR_TRY(dm.ensure(ctx, q * sizeof(uint64_t)));
  MR_TRY(di.ensure(ctx, q * sizeof(uint64_t)));
  MR_TRY(dn.ensure(ctx, q * sizeof(uint64_t)));
  MR_CUDA(ctx, cudaMemcpyAsync(dm.p, mers, q * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  MR_TRY(mr_lookup_batch_device(idx, dm.as<uint64_t>(), q, di.as<uint64_t>(), dn.as<uint64_t>()));
  MR_CUDA(ctx, cudaMemcpyAsync(index_out, di.p, q * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaMemcpyAsync(nb_out, dn.p, q * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

} // extern "C"

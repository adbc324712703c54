// Per-batch alignment pipeline on the device: seed selection + suffix-array lookup, per-read
// count threshold, hit expansion, grouping by super-read (stable radix sort), chaining ("LIS"),
// least-squares coords and filters, kmers_info, per-read ordering.  One kernel per CPU hot loop
// of the reference (SURVEY.md section 8a); every kernel cites what it replaces.
#include "align.cuh"
#include "group.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>

namespace {

// MR_TRACE=1: progress lines on stderr (which phase a stuck batch is in)
// ------------------------------------------------------------------------------------------------
// final rows, graph node arrays and the copy of both to one pinned slab: shared by mr_align_batch
// and mr_graph_batch
// ------------------------------------------------------------------------------------------------
static int setup_final_rows(mr_context* ctx, mr_workspace& ws, uint64_t Sc, coords_soa& fin) {
  memset(&fin, 0, sizeof(fin));
  MR_TRY(ws.fin_i32.ensure(ctx, Sc * 4 * 5)); MR_TRY(ws.fin_u32.ensure(ctx, Sc * 4 * 8)); MR_TRY(ws.fin_f64.ensure(ctx, Sc * 8 * 3));
  MR_TRY(ws.fin_u64.ensure(ctx, Sc * 8 * 3)); MR_TRY(ws.fin_u8.ensure(ctx, Sc * 2));
  { int32_t* b = ws.fin_i32.as<int32_t>(); fin.rs = b; fin.re = b + Sc; fin.qs = b + 2 * Sc; fin.qe = b + 3 * Sc; fin.nb_mers = b + 4 * Sc; }
  { uint32_t* b = ws.fin_u32.as<uint32_t>(); fin.pb_cons = b; fin.sr_cons = b + Sc; fin.pb_cover = b + 2 * Sc; fin.sr_cover = b + 3 * Sc;
    fin.ql = b + 4 * Sc; fin.sr = b + 5 * Sc; fin.read = b + 6 * Sc; fin.info_len = b + 7 * Sc; }
  { double* b = ws.fin_f64.as<double>(); fin.stretch = b; fin.offset = b + Sc; fin.avg_err = b + 2 * Sc; }
  { uint64_t* b = ws.fin_u64.as<uint64_t>(); fin.info_off = b; fin.chain_pos = b + Sc; }
  { uint8_t* b = ws.fin_u8.as<uint8_t>(); fin.rn = b; fin.use_bwd = b + Sc; }
  return MR_OK;
}

static int setup_graph_nodes(mr_context* ctx, mr_workspace& ws, uint64_t Sc, graph_args& GA) {
  MR_TRY(ws.node_i32.ensure(ctx, Sc * 4 * 7)); MR_TRY(ws.node_u8.ensure(ctx, Sc * 2)); MR_TRY(ws.node_f64.ensure(ctx, Sc * 8 * 5));
  { int32_t* b = ws.node_i32.as<int32_t>(); GA.lstart = b; GA.lprev = b + Sc; GA.lpath = b + 2 * Sc; GA.lunitigs = b + 3 * Sc;
    GA.component = b + 4 * Sc; GA.uf_rank = b + 5 * Sc; GA.order = b + 6 * Sc; }
  { uint8_t* b = ws.node_u8.as<uint8_t>(); GA.start_node = b; GA.end_node = b + Sc; }
  { double* b = ws.node_f64.as<double>(); GA.imp_s = b; GA.imp_e = b + Sc; GA.ord_s = b + 2 * Sc; GA.ord_e = b + 3 * Sc; GA.ord_err = b + 4 * Sc; }
  return MR_OK;
}

static int download_rows(mr_context* ctx, mr_workspace& ws, mr_result* res, const coords_soa& fin, uint32_t nreads, uint64_t S,
                         uint64_t info_total, const graph_args* GA) {
  cudaStream_t st = ctx->stream;
  const uint64_t Sc = std::max<uint64_t>(S, 1);
  auto rnd = [](uint64_t b) { return (b + 63) / 64 * 64; };
  uint64_t bytes = rnd(((uint64_t)nreads + 1) * 8) + 5 * rnd(Sc * 4) + 8 * rnd(Sc * 4) + 3 * rnd(Sc * 8) + rnd(Sc * 8) + 2 * rnd(Sc)
                   + 2 * rnd((info_total + 1) * 4) + (GA ? 2 * rnd(Sc) + 5 * rnd(Sc * 4) : 0);
  {
    std::lock_guard<std::mutex> lock(ws.pool_mutex);
    if(!ws.pinned_pool.empty()) { res->host = ws.pinned_pool.back(); ws.pinned_pool.pop_back(); }
  }
  if(!res->host) res->host = new pinned_buf;
  MR_TRY(res->host->ensure(ctx, bytes + 4096));
  char* cur = res->host->as<char>();
  auto pull = [&](const void* dsrc, uint64_t nbytes) -> const void* {
    void* dst = cur;
    cur += rnd(std::max<uint64_t>(nbytes, 1));
    if(nbytes) cudaMemcpyAsync(dst, dsrc, nbytes, cudaMemcpyDeviceToHost, st);
    return dst;
  };
  mr_result_view& v = res->view;
  v.ncoords = S;
  v.read_coords = (const uint64_t*)pull(ws.read_coords.p, ((uint64_t)nreads + 1) * 8);
  v.rs = (const int32_t*)pull(fin.rs, S * 4); v.re = (const int32_t*)pull(fin.re, S * 4);
  v.qs = (const int32_t*)pull(fin.qs, S * 4); v.qe = (const int32_t*)pull(fin.qe, S * 4);
  v.nb_mers = (const int32_t*)pull(fin.nb_mers, S * 4);
  v.pb_cons = (const uint32_t*)pull(fin.pb_cons, S * 4); v.sr_cons = (const uint32_t*)pull(fin.sr_cons, S * 4);
  v.pb_cover = (const uint32_t*)pull(fin.pb_cover, S * 4); v.sr_cover = (const uint32_t*)pull(fin.sr_cover, S * 4);
  v.ql = (const uint32_t*)pull(fin.ql, S * 4); v.sr = (const uint32_t*)pull(fin.sr, S * 4);
  v.rn = (const uint8_t*)pull(fin.rn, S); v.use_bwd = (const uint8_t*)pull(fin.use_bwd, S);
  v.stretch = (const double*)pull(fin.stretch, S * 8); v.offset = (const double*)pull(fin.offset, S * 8);
  v.avg_err = (const double*)pull(fin.avg_err, S * 8);
  v.info_off = (const uint64_t*)pull(fin.info_off, S * 8); v.info_len = (const uint32_t*)pull(fin.info_len, S * 4);
  v.kmers_info = (const int32_t*)pull(ws.kinfo.p, info_total * 4); v.bases_info = (const int32_t*)pull(ws.binfo.p, info_total * 4);
  if(GA) {
    v.start_node = (const uint8_t*)pull(GA->start_node, S); v.end_node = (const uint8_t*)pull(GA->end_node, S);
    v.lstart = (const int32_t*)pull(GA->lstart, S * 4); v.lprev = (const int32_t*)pull(GA->lprev, S * 4);
    v.lpath = (const int32_t*)pull(GA->lpath, S * 4); v.lunitigs = (const int32_t*)pull(GA->lunitigs, S * 4);
    v.component = (const int32_t*)pull(GA->component, S * 4);
  }
  MR_CUDA(ctx, cudaGetLastError());
  return MR_OK;
}

// Stamps a finished result: mr_coords_records may read its rows where they are until the next batch, and with a
// graph mr_records may too.
static void remember_rows(mr_workspace& ws, mr_result* res, const coords_soa& fin, uint32_t nreads, const graph_args* GA,
                          uint64_t S, int max_rows) {
  res->stamp = ++ws.stamp;
  ws.rows_stamp = res->stamp;
  ws.last_coords = rows_args{ nreads, S, ws.read_coords.as<uint64_t>(), ws.read_len.as<uint32_t>(), fin,
                              ws.kinfo.as<int32_t>(), ws.binfo.as<int32_t>() };
  if(!GA) return;
  ws.graph_stamp = res->stamp;
  ws.last_graph = *GA; ws.last_rows = S; ws.last_max_rows = max_rows;
}

static const bool g_trace = getenv("MR_TRACE") != nullptr;
#define MR_TRACE_MSG(...) do { if(g_trace) { fprintf(stderr, "[mr] " __VA_ARGS__); fputc('\n', stderr); fflush(stderr); } } while(0)

// ------------------------------------------------------------------------------------------------
// k-mer enumeration over one tile of one read (jf_aligner.hpp:41-52,113-123 + coarse_aligner.cc:8-15,89-102)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t base_code(char c) {
  switch(c) {
  case 'a': case 'A': return 0;
  case 'c': case 'C': return 1;
  case 'g': case 'G': return 2;
  case 't': case 'T': return 3;
  default: return 4;
  }
}

__device__ __forceinline__ bool is_ssr(uint64_t m, uint32_t k) {
  const unsigned top = 2 * (k - 1);
  const uint64_t r1 = (m >> 2) | ((m & 3) << top);
  const uint64_t r2 = (r1 >> 2) | ((r1 & 3) << top);
  return r1 == m || r2 == m;
}

struct tile_kmers {
  uint64_t m[4], rm[4];
  bool     valid[4];     // k consecutive ACGT, not a simple sequence repeat
  bool     cand[4];      // ... and still inside the first 17 bases of its N-free run: toggles `flag`
};

// Reads travel and live on the device 2-bit packed (compact_dna layout: base g at bits 2 (g % 32) of word
// g / 32, A0 C1 G2 T3) next to a 1-bit mask of the non-ACGT positions: 0.375 bytes per base instead of one
// ASCII character.  packed_reads::codes / nmask are padded by at least 4 words past the last base.
// A tile's words (at most 37 + 19) are staged in shared memory by the TMA engine (two 1-D bulk copies
// completing on an mbarrier) when the arrays are 16-byte aligned -- always, for the library's own
// buffers -- and by ordinary loads otherwise.
constexpr int kTileCodeWords = (kTile + 64 + 32) / 32 + 4;       // 39
constexpr int kTileMaskWords = (kTile + 64 + 32) / 64 + 4;       // 21
struct tile_stage {
  alignas(16) uint64_t cw[kTileCodeWords + 1];
  alignas(16) uint64_t mw[kTileMaskWords + 1];
  alignas(8)  uint64_t bar;
};
static_assert(kTileCodeWords % 2 == 1 && kTileMaskWords % 2 == 1, "the + 1 keeps the arrays a multiple of 16 bytes");

// Loads the tile's bases (plus look-back / look-ahead) into shared memory as codes; codes[] needs
// kTile + 64 bytes.  Returns whether this thread loaded a non-ACGT code (positions outside the read
// count as such).  Ends with a barrier.
__device__ __forceinline__ bool load_tile_codes(const packed_reads& pr, uint64_t rstart, uint32_t rlen,
                                                uint32_t tile_pos, uint32_t k, uint8_t* codes, tile_stage& ts) {
  const int cap = k > 18 ? (int)k : 18;        // run length is only needed up to max(k, 18)
  const int LB  = cap - (int)k;
  const int total = LB + kTile + (int)k - 1;
  // bases [gA, gB) of the batch are inside the read and inside the window
  const int64_t p0 = (int64_t)tile_pos - LB;
  const uint64_t gA = rstart + (uint64_t)(p0 > 0 ? p0 : 0);
  const int64_t pend = p0 + total;
  const uint64_t gB = rstart + (uint64_t)(pend < (int64_t)rlen ? pend : (int64_t)rlen);
  const uint64_t wa = (gA >> 5) & ~1ULL, ma = (gA >> 6) & ~1ULL;                       // 16-byte aligned starts
  const uint32_t nw = (uint32_t)((((gB + 31) >> 5) - wa + 1) & ~1ULL);                 // even word counts
  const uint32_t nm = (uint32_t)((((gB + 63) >> 6) - ma + 1) & ~1ULL);
  if(pr.tma) {
    if(threadIdx.x == 0) {
      mbar_init(&ts.bar, 1);
      mbar_expect_tx(&ts.bar, (nw + nm) * 8u);
      bulk_copy_g2s(ts.cw, pr.codes + wa, nw * 8u, &ts.bar);
      bulk_copy_g2s(ts.mw, pr.nmask + ma, nm * 8u, &ts.bar);
    }
    __syncthreads();                             // the barrier's initialisation is visible to the waiters
    mbar_wait(&ts.bar, 0);
  } else {
    for(uint32_t i = threadIdx.x; i < nw; i += kSeedThreads) ts.cw[i] = __ldg(pr.codes + wa + i);
    for(uint32_t i = threadIdx.x; i < nm; i += kSeedThreads) ts.mw[i] = __ldg(pr.nmask + ma + i);
    __syncthreads();
  }
  bool broke = false;
  for(int i = threadIdx.x; i < total; i += kSeedThreads) {
    const int64_t p = p0 + i;
    uint8_t c = 4;
    if(p >= 0 && p < (int64_t)rlen) {
      const uint64_t g = rstart + (uint64_t)p;
      const uint64_t cw = ts.cw[(g >> 5) - wa], mw = ts.mw[(g >> 6) - ma];
      c = (mw >> (g & 63)) & 1 ? (uint8_t)4 : (uint8_t)((cw >> (2 * (g & 31))) & 3);
    }
    codes[i] = c;
    broke |= c == 4;
  }
  __syncthreads();
  return broke;
}

// Enumerates the 4 consecutive k-mers owned by this thread from the codes of load_tile_codes.
__device__ __forceinline__ void tile_kmers_from_codes(uint32_t k, const uint8_t* codes, tile_kmers& t, bool every_mer = false) {
  const int cap = k > 18 ? (int)k : 18;
  const int LB  = cap - (int)k;
  const int s0 = threadIdx.x * 4;
  const uint64_t mask = (1ULL << (2 * k)) - 1;
  const unsigned top = 2 * (k - 1);
  uint64_t m = 0, rm = 0;
  for(uint32_t j = 0; j < k; ++j) {
    const uint64_t c = codes[LB + s0 + j] & 3;
    m  = (m << 2) | c;
    rm = (rm >> 2) | ((3 - c) << top);
  }
  int run = 0;
  for(int j = 0; j < cap; ++j) {
    if(codes[LB + s0 + (int)k - 1 - j] == 4) break;
    ++run;
  }
#pragma unroll
  for(int j = 0; j < 4; ++j) {
    const bool ok = run >= (int)k && (every_mer || !is_ssr(m, k));    // the fine pass takes every mer (jf_aligner.hpp:113-123)
    t.m[j] = m; t.rm[j] = rm;
    t.valid[j] = ok;
    t.cand[j]  = ok && run <= 17;
    const uint8_t c = codes[LB + s0 + j + (int)k];
    run = c == 4 ? 0 : min(run + 1, cap);
    m  = ((m << 2) | (uint64_t)(c & 3)) & mask;
    rm = (rm >> 2) | ((uint64_t)(3 - (c & 3)) << top);
  }
}

__device__ __forceinline__ void enumerate_tile(const packed_reads& bases, uint64_t rstart, uint32_t rlen,
                                               uint32_t tile_pos, uint32_t k, uint8_t* codes, tile_stage& ts, tile_kmers& t, bool every_mer = false) {
  (void)load_tile_codes(bases, rstart, rlen, tile_pos, k, codes, ts);
  tile_kmers_from_codes(k, codes, t, every_mer);
}

// ASCII bases on the device -> the packed form (the entry points that take characters); one thread
// per 64 bases: one mask word and two code words.  jf_aligner.hpp:41-52 treats every character
// outside ACGT/acgt as a break.
__global__ void __launch_bounds__(256) pack_reads_kernel(const char* __restrict__ bases, uint64_t n, uint64_t* __restrict__ codes,
                                                          uint64_t* __restrict__ nmask, uint64_t nmask_words) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(w >= nmask_words) return;
  uint64_t c0 = 0, c1 = 0, m = 0;
  const uint64_t g0 = w * 64;
  for(int j = 0; j < 64; ++j) {
    const uint64_t g = g0 + j;
    const uint8_t c = g < n ? base_code(bases[g]) : (uint8_t)0;
    const uint64_t two = c & 3;
    if(j < 32) c0 |= two << (2 * j); else c1 |= two << (2 * (j - 32));
    m |= (uint64_t)(c == 4) << j;
  }
  codes[2 * w] = c0; codes[2 * w + 1] = c1;
  nmask[w] = m;
}

// ---- k-mers straight from the packed words ---------------------------------------------------------------------
// With the reads 2-bit packed, a k-mer is a bit field: 64 bits of the code words starting at base g hold bases
// g .. g + 31 lowest first, so the k-mer as the reference numbers it (first base most significant,
// mer_sa_imp.hpp:41-47) is that field with its 2-bit groups reversed, and its reverse complement is simply the
// complemented field (base j of the k-mer lands at bits 2j, which is where the reverse complement wants the
// complement of base j).  Whether the k bases are all ACGT, and whether a run of ACGT began within the last
// 18 bases (the only k-mers that toggle the reference's every-other-k-mer flag, coarse_aligner.cc:89-102), are
// two tests on an 18-bit field of the mask words.  No per-base loop, no byte array of codes.
__device__ __forceinline__ uint64_t stage_bits(const uint64_t* w, uint64_t bit) {       // 64 bits of the array from `bit` on
  const uint32_t wi = (uint32_t)(bit >> 6), sh = (uint32_t)bit & 63;
  return sh ? (w[wi] >> sh) | (w[wi + 1] << (64 - sh)) : w[wi];
}

// Stages the words of the tile at (rstart, tile_pos) and returns where they start; ends with a barrier.
struct tile_words { uint64_t wa, ma; };          // first staged code word / mask word (indices into the batch's arrays)
__device__ __forceinline__ tile_words stage_tile_words(const packed_reads& pr, uint64_t rstart, uint32_t rlen, uint32_t tile_pos,
                                                       uint32_t k, tile_stage& ts) {
  const int cap = k > 18 ? (int)k : 18;
  const int LB  = cap - (int)k;
  const int total = LB + kTile + (int)k - 1;
  const int64_t p0 = (int64_t)tile_pos - LB;
  const uint64_t gA = rstart + (uint64_t)(p0 > 0 ? p0 : 0);
  const int64_t pend = p0 + total;
  const uint64_t gB = rstart + (uint64_t)(pend < (int64_t)rlen ? pend : (int64_t)rlen);
  tile_words tw;
  tw.wa = (gA >> 5) & ~1ULL; tw.ma = (gA >> 6) & ~1ULL;
  const uint32_t nw = (uint32_t)((((gB + 31) >> 5) - tw.wa + 1) & ~1ULL);
  const uint32_t nm = (uint32_t)((((gB + 63) >> 6) - tw.ma + 1) & ~1ULL);
  if(pr.tma) {
    if(threadIdx.x == 0) {
      mbar_init(&ts.bar, 1);
      mbar_expect_tx(&ts.bar, (nw + nm) * 8u);
      bulk_copy_g2s(ts.cw, pr.codes + tw.wa, nw * 8u, &ts.bar);
      bulk_copy_g2s(ts.mw, pr.nmask + tw.ma, nm * 8u, &ts.bar);
    }
    __syncthreads();
    mbar_wait(&ts.bar, 0);
  } else {
    for(uint32_t i = threadIdx.x; i < nw; i += kSeedThreads) ts.cw[i] = __ldg(pr.codes + tw.wa + i);
    for(uint32_t i = threadIdx.x; i < nm; i += kSeedThreads) ts.mw[i] = __ldg(pr.nmask + tw.ma + i);
    __syncthreads();
  }
  return tw;
}

// k-mer and its reverse complement at read position pos (the caller knows pos + k <= rlen)
__device__ __forceinline__ void kmer_at(const tile_stage& ts, const tile_words& tw, uint64_t g, uint32_t k, uint64_t& m, uint64_t& rm) {
  const uint64_t win = stage_bits(ts.cw, 2 * (g - 32 * tw.wa));
  const uint64_t mask = (1ULL << (2 * k)) - 1;
  m  = reverse_pairs(win) >> (64 - 2 * k);
  rm = ~win & mask;
}

// valid: k consecutive ACGT at pos, inside the read; cand: ... and a run of ACGT started within the 18 bases that end
// with the k-mer's last one (positions before the read count as non-ACGT) -- what jf_aligner.hpp:41-52's running
// `len <= 17` means.  Simple-sequence repeats are NOT excluded here.
__device__ __forceinline__ void kmer_flags(const tile_stage& ts, const tile_words& tw, uint64_t rstart, uint32_t rlen, uint32_t pos,
                                           uint32_t k, bool& valid, bool& cand) {
  valid = false; cand = false;
  if((uint64_t)pos + k > rlen) return;
  const uint64_t g = rstart + pos;
  if(k <= 18) {
    if(pos + k >= 18) {
      const uint64_t x = stage_bits(ts.mw, g + k - 18 - 64 * tw.ma) & 0x3ffffULL;      // bit t: base pos + k - 18 + t
      valid = (x >> (18 - k)) == 0;
      cand = valid && (x & ((1ULL << (18 - k)) - 1)) != 0;
    } else {                                     // the 18-base window starts before the read does
      const uint64_t x = stage_bits(ts.mw, g - 64 * tw.ma) & ((1ULL << k) - 1);
      valid = x == 0;
      cand = valid;
    }
  } else {
    valid = (stage_bits(ts.mw, g - 64 * tw.ma) & ((1ULL << k) - 1)) == 0;
  }
}

// pass 0 (only when k <= 17): number of flag-toggling k-mers per tile
__global__ void __launch_bounds__(kSeedThreads) seed_count_kernel(packed_reads bases, const uint64_t* __restrict__ read_start,
                                                                   const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                                   uint32_t k, uint32_t* __restrict__ tile_cand) {
  __shared__ tile_stage ts;
  __shared__ uint32_t total;
  if(threadIdx.x == 0) total = 0;
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs), tpos = tile_pos[blockIdx.x];
  const tile_words tw = stage_tile_words(bases, rs, rlen, tpos, k, ts);
  uint32_t c = 0;
#pragma unroll
  for(int j = 0; j < 4; ++j) {
    const uint32_t pos = tpos + threadIdx.x * 4 + j;
    bool valid, cand;
    kmer_flags(ts, tw, rs, rlen, pos, k, valid, cand);
    if(cand) {                                   // rare: only then is the k-mer itself needed (simple repeats do not toggle)
      uint64_t m, rm;
      kmer_at(ts, tw, rs + pos, k, m, rm);
      c += !is_ssr(m, k);
    }
  }
  c = __reduce_add_sync(MR_FULL_MASK, c);
  if((threadIdx.x & 31) == 0 && c) atomicAdd(&total, c);
  __syncthreads();
  if(threadIdx.x == 0) tile_cand[blockIdx.x] = total;
}

// exclusive prefix of tile_cand inside each read (the toggle persists across N breaks, coarse_aligner.cc:89)
__global__ void tile_tbase_kernel(const uint32_t* __restrict__ tile_first, uint32_t nreads,
                                  const uint32_t* __restrict__ tile_cand, uint32_t* __restrict__ tile_tbase) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if(r >= nreads) return;
  uint32_t run = 0;
  for(uint32_t t = tile_first[r]; t < tile_first[r + 1]; ++t) { tile_tbase[t] = run; run += tile_cand[t]; }
}

// Seed kernel: for every read position decides whether its k-mer is looked up
// (coarse_aligner.cc:93-102), looks up both strands (superread_parser.hpp:183-192 ->
// mer_sa_imp.hpp:369-479) and applies the max-count filter (coarse_aligner.cc:108-111).
// rec[g] = {index(m), nb(m), index(rm), nb(rm)}; size[g] = nb(m)+nb(rm) or 0 when there is no list.
// kMulti (index of several parts, index.cuh): one launch per part, each with its own rec array;
// size[g] accumulates the per-part list sizes over the launches (part_flags bit 0: first part,
// bit 1: last part) and the max-count filter is applied to the sum by the last one.
// kNib: bucket bounds come from the nibble records (index_view::nib) instead of the counts table.
// kBytes: the tails are one byte wide (k - mi <= 4), known at compile time.
// A thread owns 4 consecutive positions.  It first derives their flags (bit tests on the staged words), then
// walks them one at a time: the two strands' table reads of a position are issued together, and with 8 to 10
// warps per scheduler in flight that is all the memory parallelism the SM can use -- the first version unrolled
// all 8 lookups of a thread into 120 KB of code at 64 registers and stalled on instruction fetch (ncu:
// no_instruction) once the tables had been made to stay in the L2.
template<bool kMulti, bool kNib, bool kBytes>
__global__ void __launch_bounds__(kSeedThreads, 5) seed_lookup_kernel(index_view iv, uint32_t part_flags, packed_reads bases,
                                                                    const uint64_t* __restrict__ read_start,
                                                                    const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                                    const uint32_t* __restrict__ tile_tbase, uint32_t max_count,
                                                                    uint4* __restrict__ rec, uint32_t* __restrict__ size,
                                                                    unsigned long long* __restrict__ n_lookups,
                                                                    unsigned long long* __restrict__ n_tails,
                                                                    unsigned long long* __restrict__ n_lists,
                                                                    unsigned long long* __restrict__ n_buckets) {
  __shared__ tile_stage ts;
  __shared__ uint64_t sw[8];
  __shared__ uint32_t looked, scanned, listed, buckets;
  const uint32_t k = iv.k;
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  const uint32_t tpos = tile_pos[blockIdx.x];
  if(threadIdx.x == 0) { looked = 0; scanned = 0; listed = 0; buckets = 0; }
  const tile_words tw = stage_tile_words(bases, rs, rlen, tpos, k, ts);

  // flags of this thread's positions: bit j of keep / cand
  uint32_t keep = 0, candm = 0;
#pragma unroll
  for(int j = 0; j < 4; ++j) {
    const uint32_t pos = tpos + threadIdx.x * 4 + j;
    bool valid, cand;
    kmer_flags(ts, tw, rs, rlen, pos, k, valid, cand);
    if(valid) {
      uint64_t m, rm;
      kmer_at(ts, tw, rs + pos, k, m, rm);
      if(!is_ssr(m, k)) { keep |= 1u << j; if(cand) candm |= 1u << j; }
    }
  }
  const uint32_t ncand = __popc(candm);
  if(k <= 17 && __syncthreads_or(ncand != 0)) {
    uint64_t total;
    uint32_t seen = tile_tbase[blockIdx.x] + (uint32_t)prim::block_exclusive_scan_256(ncand, sw, total);
#pragma unroll
    for(int j = 0; j < 4; ++j) {
      if((candm >> j) & 1) {
        ++seen;                                   // flag starts at 1 and flips on every candidate:
        if((seen & 1) == 0) keep &= ~(1u << j);   // the 2nd, 4th, ... candidate of the read is skipped
      }
    }
  }

  const uint32_t tmask = iv.tail_bits >= 32 ? 0xffffffffu : ((1u << iv.tail_bits) - 1);
  uint32_t nlook = 0, ntail = 0, nlist = 0, nbucket = 0;
  const uint64_t g0 = rs + tpos + (uint64_t)threadIdx.x * 4;
#pragma unroll 1
  for(int j = 0; j < 4; ++j) {
    const uint32_t pos = tpos + threadIdx.x * 4 + j;
    if(pos >= rlen) break;
    uint4 out = make_uint4(0, 0, 0, 0);
    uint32_t sz = 0;
    if((keep >> j) & 1) {
      ++nlook;
      uint64_t mer[2];
      kmer_at(ts, tw, rs + pos, k, mer[0], mer[1]);
      uint32_t a0[2], a1[2], first[2], idx[2], nb[2];
#pragma unroll
      for(int s = 0; s < 2; ++s) bucket_bounds<kNib>(iv, (uint32_t)(mer[s] >> iv.tail_bits), a0[s], a1[s]);
#pragma unroll
      for(int s = 0; s < 2; ++s) first[s] = a0[s] != a1[s] ? tail_word(iv, kBytes ? a0[s] >> 2 : tail_word_of(iv, a0[s])) : 0u;
#pragma unroll
      for(int s = 0; s < 2; ++s) {
        idx[s] = 0; nb[s] = 0;
        if(a0[s] != a1[s]) {
          const uint32_t tt = (uint32_t)mer[s] & tmask;
          uint32_t lo, hi;
          ntail += a1[s] - a0[s] <= 64 ? a1[s] - a0[s] : 2 * (32 - __clz(a1[s] - a0[s]));   // entries a scan / two binary searches touch
          ++nbucket;
          if(kBytes) bucket_range_bytes(iv, a0[s], a1[s], tt, first[s], lo, hi);
          else       bucket_range(iv, a0[s], a1[s], tt, first[s], lo, hi);
          if(hi != lo && (mer[s] & 3) == 0)
            for(uint32_t q = 0; q < iv.nshort; ++q) lo += iv.short_key[q] == mer[s];
          nb[s] = hi - lo; idx[s] = nb[s] ? lo : 0;
        }
      }
      const uint32_t total = nb[0] + nb[1];
      if(kMulti || (total != 0 && !(max_count && total >= max_count))) {
        out = make_uint4(idx[0], nb[0], idx[1], nb[1]);
        sz = total;
      }
    }
    // streaming stores (evict-first): the output must not push the index tables out of L2
    if(kMulti) {
      if(!(part_flags & 1)) sz += size[g0 + j];
      if((part_flags & 2) && max_count && sz >= max_count) sz = 0;
    }
    // expand_kernel reads rec only where size != 0 (a one-part index): positions without a list
    // (most of them) write 4 bytes instead of 20
    if(kMulti || sz) __stcs(rec + g0 + j, out);
    __stcs(size + g0 + j, sz);
    if((!kMulti || (part_flags & 2)) && sz) ++nlist;
  }
  if(kMulti && !(part_flags & 1)) nlook = 0;          // a k-mer is counted once, not once per part
  nlook = __reduce_add_sync(MR_FULL_MASK, nlook); ntail = __reduce_add_sync(MR_FULL_MASK, ntail);
  nlist = __reduce_add_sync(MR_FULL_MASK, nlist); nbucket = __reduce_add_sync(MR_FULL_MASK, nbucket);
  if((threadIdx.x & 31) == 0) {
    if(nlook) atomicAdd(&looked, nlook);
    if(ntail) atomicAdd(&scanned, ntail);
    if(nlist) atomicAdd(&listed, nlist);
    if(nbucket) atomicAdd(&buckets, nbucket);
  }
  __syncthreads();
  if(threadIdx.x == 0) {
    if(looked) atomicAdd(n_lookups, (unsigned long long)looked);
    if(scanned) atomicAdd(n_tails, (unsigned long long)scanned);
    if(listed) atomicAdd(n_lists, (unsigned long long)listed);
    if(buckets) atomicAdd(n_buckets, (unsigned long long)buckets);
  }
}

// ------------------------------------------------------------------------------------------------
// per-read count threshold (coarse_aligner.cc:117-131): smallest t with #{size <= t} > round(0.99 #lists),
// found by a most-significant-digit-first radix select; lists above it get size 0.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) read_threshold_kernel(const uint64_t* __restrict__ read_start, uint32_t nbits,
                                                              uint32_t* __restrict__ size, uint32_t* __restrict__ thr_out) {
  __shared__ uint32_t hist[2048];
  __shared__ uint64_t sw[8];
  __shared__ uint32_t sh_bin, sh_before, sh_count;
  const uint32_t r = blockIdx.x;
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  uint32_t* sz = size + rs;
  if(threadIdx.x == 0) sh_count = 0;
  __syncthreads();
  uint32_t mine = 0;
  for(uint32_t i = threadIdx.x; i < rlen; i += 256) mine += sz[i] != 0;
  if(mine) atomicAdd(&sh_count, mine);
  __syncthreads();
  const uint32_t L = sh_count;
  const double   scaled = (double)L * 0.99;
  const uint32_t sum_thresh = (uint32_t)round(scaled);
  if(L == 0 || sum_thresh >= L) { if(threadIdx.x == 0) thr_out[r] = 0xffffffffu; return; }
  uint32_t kth = sum_thresh + 1, prefix = 0, remaining = nbits;
  while(remaining > 0) {
    const uint32_t d = remaining < 11 ? remaining : 11, shift = remaining - d;
    for(int i = threadIdx.x; i < 2048; i += 256) hist[i] = 0;
    __syncthreads();
    for(uint32_t i = threadIdx.x; i < rlen; i += 256) {
      const uint32_t v = sz[i];
      if(v != 0 && (remaining >= 32 || (v >> remaining) == prefix)) atomicAdd(&hist[(v >> shift) & ((1u << d) - 1)], 1u);
    }
    __syncthreads();
    uint32_t local[8], s = 0;
#pragma unroll
    for(int j = 0; j < 8; ++j) { local[j] = hist[threadIdx.x * 8 + j]; s += local[j]; }
    uint64_t total;
    uint32_t before = (uint32_t)prim::block_exclusive_scan_256(s, sw, total);
    if(before < kth && kth <= before + s) {
#pragma unroll
      for(int j = 0; j < 8; ++j) {
        if(kth <= before + local[j]) { sh_bin = threadIdx.x * 8 + j; sh_before = before; break; }
        before += local[j];
      }
    }
    __syncthreads();
    kth -= sh_before;
    prefix = (prefix << d) | sh_bin;
    remaining = shift;
    __syncthreads();
  }
  if(threadIdx.x == 0) thr_out[r] = prefix;
  for(uint32_t i = threadIdx.x; i < rlen; i += 256) if(sz[i] > prefix) sz[i] = 0;
}

// ------------------------------------------------------------------------------------------------
// hit expansion (coarse_aligner.cc:127-138 + pos_iterator, superread_parser.hpp:110-134):
// every SA entry of a kept list becomes (key = read<<32 | super-read, payload = pb offset, signed
// super-read offset); entries whose k-mer straddles two super-reads get super-read == nseq.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void emit_hit(const index_view& iv, uint32_t read, uint32_t pb_off, uint32_t sa_rank, bool minus,
                                         uint64_t slot, uint64_t* __restrict__ keys, uint64_t* __restrict__ pays,
                                         uint32_t& n_bad) {
  uint32_t sr, off;
  bool inside;
  if(iv.saloc) {
    const uint2 l = __ldg(iv.saloc + sa_rank);
    sr = l.x; off = l.y;
    inside = sr != 0xffffffffu;
  } else inside = index_locate(iv, __ldg(iv.sa + sa_rank), sr, off);
  if(inside) {
    const int32_t soff = minus ? -(int32_t)off : (int32_t)off;
    keys[slot] = ((uint64_t)read << 32) | (iv.sr_base + sr);
    pays[slot] = (uint64_t)pb_off | ((uint64_t)(uint32_t)soff << 32);
  } else {
    keys[slot] = ((uint64_t)read << 32) | iv.nseq_all;
    pays[slot] = 0;
    ++n_bad;
  }
}

// hits per tile (lists that survived the count threshold); their exclusive scan gives every tile its
// slice of the hit arrays, and expand_kernel redoes the scan inside the tile: no per-position
// offset array (8 B x read bases written and read back) is needed
__global__ void __launch_bounds__(kSeedThreads) tile_hits_kernel(const uint64_t* __restrict__ read_start,
                                                                  const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                                  const uint32_t* __restrict__ size, uint32_t* __restrict__ tile_hits,
                                                                  unsigned long long* __restrict__ overflow) {
  __shared__ uint64_t sw[8];
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  const uint32_t tpos = tile_pos[blockIdx.x];
  uint32_t s = 0;
#pragma unroll
  for(int it = 0; it < kTile / kSeedThreads; ++it) {
    const uint32_t pos = tpos + it * kSeedThreads + threadIdx.x;
    if(pos < rlen) s += __ldcs(size + rs + pos);
  }
  uint64_t total;
  (void)prim::block_exclusive_scan_256(s, sw, total);
  // a tile total of 2^32 or more (only without --max-count, on a degenerate text) must not wrap: the
  // batch is refused (MR_ELIMIT) and the caller halves it
  if(threadIdx.x == 0) {
    tile_hits[blockIdx.x] = total > 0xffffffffULL ? 0xffffffffu : (uint32_t)total;
    if(total > 0xffffffffULL) atomicAdd(overflow, 1ULL);
  }
}

// kMulti: rec holds one array per part, rec_stride entries apart; a list is the concatenation of its
// per-part lists (forward then backward entries of part 0, of part 1, ...), more_views[p - 1] is
// the view of part p.
template<bool kMulti>
__global__ void __launch_bounds__(kSeedThreads) expand_kernel(index_view iv, const index_view* __restrict__ more_views, uint32_t nparts,
                                                               uint64_t rec_stride, const uint64_t* __restrict__ read_start,
                                                               const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                               const uint4* __restrict__ rec, const uint32_t* __restrict__ size,
                                                               const uint64_t* __restrict__ tile_off,
                                                               uint64_t* __restrict__ keys, uint64_t* __restrict__ pays,
                                                               unsigned long long* __restrict__ n_invalid) {
  __shared__ uint64_t sw[8];
  __shared__ uint32_t s_off[kSeedThreads];
  __shared__ uint4    s_rec[kSeedThreads];
  uint64_t run = tile_off[blockIdx.x];
  if(tile_off[blockIdx.x + 1] == run) return;          // nothing in this tile
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  const uint32_t tpos = tile_pos[blockIdx.x];
  uint32_t n_bad = 0;
  for(int it = 0; it < kTile / kSeedThreads; ++it) {
    const uint32_t pos = tpos + it * kSeedThreads + threadIdx.x;
    uint32_t sz = 0;
    uint4 rc = make_uint4(0, 0, 0, 0);
    if(pos < rlen) {
      sz = __ldcs(size + rs + pos);
      if(sz) rc = __ldcs(rec + rs + pos);
    }
    uint64_t in_iter;
    s_off[threadIdx.x] = (uint32_t)prim::block_exclusive_scan_256(sz, sw, in_iter);   // 256 lists below max-count: fits 32 bits
    s_rec[threadIdx.x] = rc;
    __syncthreads();
    // one thread per HIT, not per list: thread h finds the position whose list holds hit h (the last
    // position whose offset is <= h; empty lists share their offset with the next one), so the loads
    // of different hits are independent and the stores of a warp are 32 consecutive slots
    for(uint32_t h = threadIdx.x; h < (uint32_t)in_iter; h += kSeedThreads) {
      uint32_t lo = 0, hi = kSeedThreads;
      while(hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if(s_off[mid] <= h) lo = mid; else hi = mid; }
      uint4 c = s_rec[lo];
      uint32_t j = h - s_off[lo];
      if(kMulti) {
        uint32_t part = 0;
        while(j >= c.y + c.w && part + 1 < nparts) {       // the list continues in the next part
          j -= c.y + c.w;
          ++part;
          c = __ldg(rec + part * rec_stride + rs + tpos + it * kSeedThreads + lo);
        }
        const bool minus = j >= c.y;
        emit_hit(part ? more_views[part - 1] : iv, r, tpos + it * kSeedThreads + lo + 1, minus ? c.z + (j - c.y) : c.x + j, minus,
                 run + h, keys, pays, n_bad);
        continue;
      }
      const bool minus = j >= c.y;
      emit_hit(iv, r, tpos + it * kSeedThreads + lo + 1, minus ? c.z + (j - c.y) : c.x + j, minus, run + h, keys, pays, n_bad);
    }
    run += in_iter;
    __syncthreads();
  }
  if(n_bad) atomicAdd(n_invalid, (unsigned long long)n_bad);
}

// ------------------------------------------------------------------------------------------------
// fine pass (-F, fine_aligner.hpp:49-58 + fine_aligner.cc:7-51): every coarse row opens a window on
// its read; all hits of the shorter mer that land on the row's super-read inside the window are
// chained with accept-all predicates and give the row's new coords.
// ------------------------------------------------------------------------------------------------
// windows (prime_frags_pos) + the (read, super-read) -> row table, unsorted
__global__ void __launch_bounds__(256) fine_windows_kernel(uint64_t S, survivors sv, const uint64_t* __restrict__ read_start, uint32_t kk,
                                                            uint64_t* __restrict__ wkey, uint32_t* __restrict__ wrow,
                                                            double* __restrict__ wbegin, double* __restrict__ wend,
                                                            uint32_t* __restrict__ gread, uint32_t* __restrict__ gsr, uint32_t* __restrict__ giter) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= S) return;
  const uint32_t read = sv.read[i], sr = sv.sr[i];
  const double stretch = sv.stretch[i], offset = sv.offset[i], err = sv.avg_err[i];
  const double rl = (double)(read_start[read + 1] - read_start[read]);
  const double s1 = stretch + offset;
  wbegin[i] = fmax(0.0, s1 - err);
  const double t = stretch * (double)sv.ql[i];
  const double e1 = t + offset;
  const double e2 = e1 + err;
  wend[i] = fmin(rl, e2 - (double)kk);
  wkey[i] = ((uint64_t)read << 32) | sr;
  wrow[i] = (uint32_t)i;
  gread[i] = read; gsr[i] = sr; giter[i] = sv.iter[i];
}

// lookups of every kk-mer of the reads: rec = {index(m), nb(m), index(rm), nb(rm)}, size = nb(m) + nb(rm)
__global__ void __launch_bounds__(kSeedThreads) fine_seed_kernel(index_view iv, bool first_part, uint32_t kk, packed_reads bases,
                                                                  const uint64_t* __restrict__ read_start,
                                                                  const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                                  const uint64_t* __restrict__ table_off,
                                                                  uint4* __restrict__ rec, uint32_t* __restrict__ size) {
  __shared__ uint8_t codes[kTile + 64];
  __shared__ tile_stage ts;
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  const uint32_t tpos = tile_pos[blockIdx.x];
  const bool has_rows = table_off[r + 1] != table_off[r];        // a read without coarse rows has no window
  tile_kmers t;
  enumerate_tile(bases, rs, rlen, tpos, kk, codes, ts, t, true);
  const uint64_t g0 = rs + tpos + (uint64_t)threadIdx.x * 4;
#pragma unroll
  for(int j = 0; j < 4; ++j) {
    const uint32_t pos = tpos + threadIdx.x * 4 + j;
    if(pos >= rlen) continue;
    uint4 out = make_uint4(0, 0, 0, 0);
    if(has_rows && t.valid[j]) {
      index_lookup_prefix(iv, t.m[j], kk, out.x, out.y);
      index_lookup_prefix(iv, t.rm[j], kk, out.z, out.w);
    }
    __stcs(rec + g0 + j, out);
    __stcs(size + g0 + j, (first_part ? 0u : size[g0 + j]) + out.y + out.w);      // one launch per index part
  }
}

// EMIT = false: counts, per tile and per row, the hits that fall into a window; EMIT = true: writes
// them (key = row, payload = pb offset | signed super-read offset << 32) in emission order
// (read position, forward range before reverse range, suffix-array order).
template<bool EMIT>
__global__ void __launch_bounds__(kSeedThreads) fine_expand_kernel(index_view iv, const index_view* __restrict__ more_views, uint32_t nparts,
                                                                    uint64_t rec_stride, uint32_t kk, const uint64_t* __restrict__ read_start,
                                                                    const uint32_t* __restrict__ tile_read, const uint32_t* __restrict__ tile_pos,
                                                                    const uint4* __restrict__ rec, const uint32_t* __restrict__ size,
                                                                    const uint64_t* __restrict__ table_off, const uint64_t* __restrict__ tkey,
                                                                    const uint32_t* __restrict__ trow,
                                                                    const double* __restrict__ wbegin, const double* __restrict__ wend,
                                                                    uint32_t* __restrict__ tile_cnt, const uint64_t* __restrict__ tile_off,
                                                                    uint32_t* __restrict__ row_cnt,
                                                                    uint64_t* __restrict__ keys, uint64_t* __restrict__ pays) {
  __shared__ uint64_t sw[8];
  __shared__ uint32_t s_off[kSeedThreads];
  __shared__ uint4    s_rec[kSeedThreads];
  const uint32_t r = tile_read[blockIdx.x];
  const uint64_t t0 = table_off[r], t1 = table_off[r + 1];
  if(t0 == t1) { if(!EMIT && threadIdx.x == 0) tile_cnt[blockIdx.x] = 0; return; }
  if(EMIT && tile_off[blockIdx.x + 1] == tile_off[blockIdx.x]) return;
  const uint64_t rs = read_start[r];
  const uint32_t rlen = (uint32_t)(read_start[r + 1] - rs);
  const uint32_t tpos = tile_pos[blockIdx.x];
  uint64_t run = EMIT ? tile_off[blockIdx.x] : 0;
  for(int it = 0; it < kTile / kSeedThreads; ++it) {
    const uint32_t pos = tpos + it * kSeedThreads + threadIdx.x;
    uint32_t sz = 0;
    uint4 rc = make_uint4(0, 0, 0, 0);
    if(pos < rlen) {
      sz = __ldcs(size + rs + pos);
      if(sz) rc = __ldcs(rec + rs + pos);
    }
    uint64_t raw_total;
    s_off[threadIdx.x] = (uint32_t)prim::block_exclusive_scan_256(sz, sw, raw_total);
    s_rec[threadIdx.x] = rc;
    __syncthreads();
    for(uint32_t base = 0; base < (uint32_t)raw_total; base += kSeedThreads) {
      const uint32_t h = base + threadIdx.x;
      uint32_t nmatch = 0, first = 0, sr = 0, off = 0, pb_off = 0;
      bool minus = false;
      if(h < (uint32_t)raw_total) {
        uint32_t lo = 0, hi = kSeedThreads;
        while(hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if(s_off[mid] <= h) lo = mid; else hi = mid; }
        uint4 c = s_rec[lo];
        uint32_t j = h - s_off[lo];
        uint32_t part = 0;
        while(j >= c.y + c.w && part + 1 < nparts) {        // the list continues in the next index part
          j -= c.y + c.w;
          ++part;
          c = __ldg(rec + part * rec_stride + rs + tpos + it * kSeedThreads + lo);
        }
        const index_view& pv = part ? more_views[part - 1] : iv;
        minus = j >= c.y;
        pb_off = tpos + it * kSeedThreads + lo + 1;
        const uint32_t x = __ldg(pv.sa + (minus ? c.z + (j - c.y) : c.x + j));
        if(index_locate_k(pv, x, kk, sr, off)) {
          sr += pv.sr_base;
          // rows of (read, sr) in the table: equal keys are contiguous
          const uint64_t want = ((uint64_t)r << 32) | sr;
          uint64_t a = t0, b = t1;
          while(a < b) { const uint64_t mid = (a + b) >> 1; if(tkey[mid] < want) a = mid + 1; else b = mid; }
          first = (uint32_t)a;
          for(uint64_t q = a; q < t1 && tkey[q] == want; ++q) {
            const uint32_t row = trow[q];
            const double p = (double)pb_off;
            if(p >= wbegin[row] && p <= wend[row]) {
              ++nmatch;
              if(!EMIT) atomicAdd(row_cnt + row, 1u);
            }
          }
        }
      }
      uint64_t chunk_total;
      const uint64_t mine = prim::block_exclusive_scan_256(nmatch, sw, chunk_total);
      if(EMIT && nmatch) {
        const uint64_t want = ((uint64_t)r << 32) | sr;
        const int32_t soff = minus ? -(int32_t)off : (int32_t)off;
        uint64_t slot = run + mine;
        for(uint64_t q = first; q < t1 && tkey[q] == want; ++q) {
          const uint32_t row = trow[q];
          const double p = (double)pb_off;
          if(p >= wbegin[row] && p <= wend[row]) {
            keys[slot] = row;
            pays[slot] = (uint64_t)pb_off | ((uint64_t)(uint32_t)soff << 32);
            ++slot;
          }
        }
      }
      run += chunk_total;
    }
    __syncthreads();
  }
  if(!EMIT && threadIdx.x == 0) tile_cnt[blockIdx.x] = (uint32_t)run;
}

// ------------------------------------------------------------------------------------------------
// group heads: one group per (read, super-read) present in the sorted hits (frags_pos_type,
// coarse_aligner.hpp:14, as a segmented array instead of an unordered_map of vectors)
// ------------------------------------------------------------------------------------------------
struct head_flag {
  const uint64_t* keys; uint32_t nseq;
  __device__ uint64_t operator()(uint64_t i) const {
    const uint64_t k = keys[i];
    return ((uint32_t)k < nseq) && (i == 0 || keys[i - 1] != k);
  }
};
// the per-read sort (group.cu) leaves one byte per hit
struct head_byte {
  const uint8_t* head;
  __device__ uint64_t operator()(uint64_t i) const { return head[i]; }
};


// ------------------------------------------------------------------------------------------------
// kmers_info / bases_info per surviving coords: compute_kmers_info::add_mer (pb_aligner.cc:84-143),
// one thread per coords row walking its chain.
// ------------------------------------------------------------------------------------------------
struct info_args {
  uint64_t n;
  const uint64_t* chain_pos; const int32_t* nb_mers; const uint32_t* sr; const uint8_t* use_bwd; const uint32_t* ql;
  const uint64_t* info_off; uint32_t* info_len;
  const uint64_t* chain_pay;
  const uint32_t* unitig_ids; const uint64_t* unitig_off; const int32_t* unitig_len; uint32_t n_unitigs;
  uint32_t k, unitigs_k;
  int32_t* kinfo; int32_t* binfo;
};

// One THREAD per coords row walking its chain (pairs stored in chain order by the chaining kernels):
// 32 rows share every instruction.  Counters and unitig lengths of paths of up to kInfoLocal
// unitigs live in thread-local arrays (L1), so the sequential walk pays ~L1 latency per hit; longer
// paths work directly on the output slice.
constexpr int kInfoLocal = 24;

// Elements [t_begin, t_end) of the chain.  A segment that does not start at 0 first puts itself in the
// state the sequential walk has after element t_begin - 1: previous position = that element's, current
// unitig = the first one the element's mer ends in (the walk only moves forward and the ends of the
// unitigs increase along the path -- the caller checks that -- so this is where the walk stands).
// The pending counters start at 0: sums are what is stored, every segment adds its share.
template<bool LOCAL>
__device__ __forceinline__ bool kmers_info_walk(const info_args& A, uint64_t i, uint32_t nu, int32_t* mers, int32_t* bases,
                                                const int32_t* ulen_tab, uint32_t t_begin = 0, uint32_t t_end = 0xffffffffu) {
  const uint32_t sr = A.sr[i];
  const bool bwd = A.use_bwd[i];
  const uint64_t u0 = A.unitig_off[sr];
  auto ulen = [&](uint32_t t) -> int {               // -1: invalid id or past the end of the path
    if(t >= nu) return -1;
    if(LOCAL) return ulen_tab[t];
    const uint32_t id = (bwd ? A.unitig_ids[u0 + nu - 1 - t] : A.unitig_ids[u0 + t]) >> 1;
    return id < A.n_unitigs ? A.unitig_len[id] : -1;
  };
  const int K = (int)A.k, UK = (int)A.unitigs_k;
  const uint64_t* cp = A.chain_pay + A.chain_pos[i];
  const uint32_t nb = (uint32_t)A.nb_mers[i];
  const int64_t ql = A.ql[i];
  uint32_t cunitig = 0;
  int cend = ulen(0), prev_pos = -K;
  int cur_mers = 0, cur_bases = 0;                    // pending additions to mers/bases[2 * cunitig]
  const bool fwd_align = (int32_t)(uint32_t)(cp[0] >> 32) > 0;
  if(t_end > nb) t_end = nb;
  if(t_begin != 0) {
    const int32_t so = (int32_t)(uint32_t)(cp[t_begin - 1] >> 32);
    const int pos = fwd_align ? so : (int)(ql + so - K + 2);
    prev_pos = pos < 0 ? -pos : pos;
    while(prev_pos + K > cend + 1) {
      const int ul = ulen(++cunitig);
      if(ul < 0) return true;                      // the segment that owns that element reports the error
      cend += ul - UK + 1;
    }
  }
  uint64_t nxt = cp[t_begin];
  for(uint32_t t = t_begin; t < t_end; ++t) {
    const uint64_t p = nxt;
    if(t + 1 < t_end) nxt = cp[t + 1];
    const int32_t so = (int32_t)(uint32_t)(p >> 32);
    const int pos = fwd_align ? so : (int)(ql + so - K + 2);
    const int sr_pos = pos < 0 ? -pos : pos;
    const int new_bases = min(K, sr_pos - prev_pos);
    while(sr_pos + K > cend + 1) {
      if(cend >= sr_pos) {
        if(cunitig >= nu - 1) return false;
        const int nbb = cend - max(sr_pos, prev_pos + K) + 1;
        cur_bases += nbb;
        bases[2 * cunitig + 1] += nbb;
      }
      mers[2 * cunitig] += cur_mers; bases[2 * cunitig] += cur_bases;
      cur_mers = 0; cur_bases = 0;
      const int ul = ulen(++cunitig);
      if(ul < 0) return false;
      cend += ul - UK + 1;
    }
    ++cur_mers;
    cur_bases += new_bases;
    int cendi = cend;
    for(uint32_t v = cunitig; v < nu - 1 && sr_pos + K > cendi - UK + 1; ++v) {
      const int full_mer = sr_pos + UK > cendi + 1;
      mers[2 * v + 1] += full_mer;
      mers[2 * v + 2] += full_mer;
      const int nbb = min(new_bases, sr_pos + K - cendi + UK - 2);
      bases[2 * v + 1] += nbb;
      bases[2 * v + 2] += nbb;
      const int ul = ulen(v + 1);
      if(ul >= 0) cendi += ul - UK + 1;
      else return false;
    }
    prev_pos = sr_pos;
  }
  mers[2 * cunitig] += cur_mers; bases[2 * cunitig] += cur_bases;
  return true;
}

// One WARP per coords row.  The chain is cut into pieces of kInfoPiece hits; lane l of the warp takes
// piece l of every run of 32 pieces, so the warp reads 32 x kInfoPiece consecutive pairs at once
// (coalesced, all loads in flight together) instead of 32 threads each following a private stream one
// dependent load at a time.  Every piece starts in the state the sequential walk has there (see
// kmers_info_walk) and adds its counts to the row's counters in shared memory.
constexpr int kInfoPiece = 8;

__global__ void __launch_bounds__(128) kmers_info_kernel(info_args A) {
  __shared__ int32_t s_ul[4][kInfoLocal], s_m[4][2 * kInfoLocal], s_b[4][2 * kInfoLocal];
  const unsigned lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint64_t i = (uint64_t)blockIdx.x * 4 + wib;
  if(i >= A.n) return;
  const uint32_t ilen = A.info_len[i];
  if(ilen == 0) return;
  int32_t* gm = A.kinfo + A.info_off[i];
  int32_t* gb = A.binfo + A.info_off[i];
  const uint32_t sr = A.sr[i];
  const uint64_t u0 = A.unitig_off[sr];
  const uint32_t nu = (uint32_t)(A.unitig_off[sr + 1] - u0);
  if(nu > (uint32_t)kInfoLocal) {                  // long unitig paths: one thread, counters in the output slice itself
    if(lane == 0) {
      for(uint32_t j = 0; j < ilen; ++j) { gm[j] = 0; gb[j] = 0; }
      if(!kmers_info_walk<false>(A, i, nu, gm, gb, nullptr)) A.info_len[i] = 0;
    }
    return;
  }
  int32_t *ul = s_ul[wib], *sm = s_m[wib], *sb = s_b[wib];
  const int K = (int)A.k, UK = (int)A.unitigs_k;
  const bool bwd = A.use_bwd[i];
  bool bad_step = false;
  if(lane < nu) {
    const uint32_t id = (bwd ? A.unitig_ids[u0 + nu - 1 - lane] : A.unitig_ids[u0 + lane]) >> 1;
    const int len = id < A.n_unitigs ? A.unitig_len[id] : -1;
    ul[lane] = len;
    bad_step = lane != 0 && len >= 0 && len - UK + 1 < 0;
  }
  for(uint32_t j = lane; j < ilen; j += 32) { sm[j] = 0; sb[j] = 0; }
  const bool increasing = !__any_sync(MR_FULL_MASK, bad_step);   // unitig ends increase along the path (always, for real k-unitigs)
  __syncwarp();
  if(!increasing) {                                // odd unitig lengths: the plain sequential walk
    bool ok = true;
    if(lane == 0) ok = kmers_info_walk<true>(A, i, nu, sm, sb, ul);
    ok = __shfl_sync(MR_FULL_MASK, (int)ok, 0) != 0;
    __syncwarp();
    if(ok) { for(uint32_t j = lane; j < ilen; j += 32) { gm[j] = sm[j]; gb[j] = sb[j]; } }
    else if(lane == 0) A.info_len[i] = 0;
    return;
  }
  const uint64_t* cp = A.chain_pay + A.chain_pos[i];
  const uint32_t nb = (uint32_t)A.nb_mers[i];
  const int64_t ql = A.ql[i];
  const bool fwd_align = (int32_t)(uint32_t)(cp[0] >> 32) > 0;
  auto position = [&](uint64_t p) -> int {
    const int32_t so = (int32_t)(uint32_t)(p >> 32);
    const int pos = fwd_align ? so : (int)(ql + so - K + 2);
    return pos < 0 ? -pos : pos;
  };
  auto ulen = [&](uint32_t t) -> int { return t < nu ? ul[t] : -1; };
  bool failed = false;
  for(uint32_t base = 0; base < nb; base += 32 * kInfoPiece) {
    const uint32_t t0 = base + lane * kInfoPiece;
    uint64_t q[kInfoPiece], before = 0;
#pragma unroll
    for(int j = 0; j < kInfoPiece; ++j) q[j] = t0 + j < nb ? cp[t0 + j] : 0;
    if(t0 != 0 && t0 < nb) before = cp[t0 - 1];
    if(t0 < nb && !failed) {
      uint32_t cunitig = 0;
      int cend = ulen(0), prev_pos = -K, cur_mers = 0, cur_bases = 0;
      bool ok = true;
      if(t0 != 0) {
        prev_pos = position(before);
        while(prev_pos + K > cend + 1) {
          const int len = ulen(++cunitig);
          if(len < 0) break;                       // the piece that owns that hit reports the error
          cend += len - UK + 1;
        }
        ok = cunitig < nu;
      }
#pragma unroll
      for(int j = 0; j < kInfoPiece; ++j) {
        if(!ok || t0 + j >= nb) break;
        const int sr_pos = position(q[j]);
        const int new_bases = min(K, sr_pos - prev_pos);
        while(sr_pos + K > cend + 1) {
          if(cend >= sr_pos) {
            if(cunitig >= nu - 1) { failed = true; break; }
            const int nbb = cend - max(sr_pos, prev_pos + K) + 1;
            cur_bases += nbb;
            if(nbb) atomicAdd(sb + 2 * cunitig + 1, nbb);
          }
          if(cur_mers) atomicAdd(sm + 2 * cunitig, cur_mers);
          if(cur_bases) atomicAdd(sb + 2 * cunitig, cur_bases);
          cur_mers = 0; cur_bases = 0;
          const int len = ulen(++cunitig);
          if(len < 0) { failed = true; break; }
          cend += len - UK + 1;
        }
        if(failed) break;
        ++cur_mers;
        cur_bases += new_bases;
        int cendi = cend;
        for(uint32_t v = cunitig; v < nu - 1 && sr_pos + K > cendi - UK + 1; ++v) {
          const int full_mer = sr_pos + UK > cendi + 1;
          if(full_mer) { atomicAdd(sm + 2 * v + 1, 1); atomicAdd(sm + 2 * v + 2, 1); }
          const int nbb = min(new_bases, sr_pos + K - cendi + UK - 2);
          if(nbb) { atomicAdd(sb + 2 * v + 1, nbb); atomicAdd(sb + 2 * v + 2, nbb); }
          const int len = ulen(v + 1);
          if(len >= 0) cendi += len - UK + 1;
          else { failed = true; break; }
        }
        if(failed) break;
        prev_pos = sr_pos;
      }
      if(!failed && ok) {
        if(cur_mers) atomicAdd(sm + 2 * cunitig, cur_mers);
        if(cur_bases) atomicAdd(sb + 2 * cunitig, cur_bases);
      }
    }
    failed = __any_sync(MR_FULL_MASK, failed);
    if(failed) break;
  }
  __syncwarp();
  if(!failed) { for(uint32_t j = lane; j < ilen; j += 32) { gm[j] = sm[j]; gb[j] = sb[j]; } }
  else if(lane == 0) A.info_len[i] = 0;      // the reference clears both vectors on error
}

// ------------------------------------------------------------------------------------------------
// per-read ordering of the coords rows: (rs, re, ql) as create_mega_reads.cc:69-77 /
// pb_aligner.hpp:142-145, ties by super-read index (canonical; the reference's order there
// depends on unordered_map iteration and an unstable sort)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bucket_rows_kernel(uint64_t n, const uint32_t* __restrict__ read, const uint64_t* __restrict__ read_coords,
                                                           uint32_t* __restrict__ cursor, uint32_t* __restrict__ slot) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n) return;
  const uint32_t r = read[i];
  slot[read_coords[r] + atomicAdd(cursor + r, 1u)] = (uint32_t)i;
}

// Order of a read's rows by (rs, re, ql, super-read, iteration) -- create_mega_reads.cc:69-77 plus the
// canonical tie rule -- by counting, for every row, the rows that come before it.  The five keys of a
// row are first gathered next to each other in slot order (row_keys_kernel), so that the quadratic
// loop reads one contiguous, warp-uniform stream; a read with many rows (repeats: thousands) gets a
// whole CTA, the usual read (a dozen rows) one warp.
struct row_key { int32_t rs, re; uint32_t ql, sr, iter; };
__device__ __forceinline__ bool row_key_less(const row_key& b, const row_key& a) {
  return b.rs < a.rs || (b.rs == a.rs && (b.re < a.re || (b.re == a.re && (b.ql < a.ql || (b.ql == a.ql && (b.sr < a.sr || (b.sr == a.sr && b.iter < a.iter)))))));
}
__global__ void __launch_bounds__(256) row_keys_kernel(uint64_t S, const uint32_t* __restrict__ slot,
                                                       const int32_t* __restrict__ rs, const int32_t* __restrict__ re,
                                                       const uint32_t* __restrict__ ql, const uint32_t* __restrict__ sr,
                                                       const uint32_t* __restrict__ iter, int4* __restrict__ k4, uint32_t* __restrict__ k5) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= S) return;
  const uint32_t me = slot[i];
  k4[i] = make_int4(rs[me], re[me], (int)ql[me], (int)sr[me]);
  k5[i] = iter[me];
}
__global__ void __launch_bounds__(128) rank_rows_kernel(uint32_t nreads, const uint64_t* __restrict__ read_coords, const uint32_t* __restrict__ slot,
                                                         const int4* __restrict__ k4, const uint32_t* __restrict__ k5,
                                                         uint32_t warp_max, uint32_t* __restrict__ order) {
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, first = threadIdx.x & 31;
  if(r >= nreads) return;
  const uint64_t b = read_coords[r];
  const uint32_t c = (uint32_t)(read_coords[r + 1] - b);
  if(c > warp_max) return;
  for(uint32_t e = first; e < c; e += 32) {
    const int4 a4 = k4[b + e];
    const row_key a = { a4.x, a4.y, (uint32_t)a4.z, (uint32_t)a4.w, k5[b + e] };
    uint32_t rank = 0;
    for(uint32_t f = 0; f < c; ++f) {
      const int4 o4 = __ldg(k4 + b + f);
      const row_key o = { o4.x, o4.y, (uint32_t)o4.z, (uint32_t)o4.w, __ldg(k5 + b + f) };
      rank += row_key_less(o, a);
    }
    order[b + rank] = slot[b + e];
  }
}

// A read with many rows (repeats: hundreds to thousands): one CTA.  Up to sort_cap rows the keys go to
// shared memory and the row indices are sorted there (bitonic network; the five keys of two rows never tie
// completely -- the super-read and the --max-match round tell them apart); above, the rows are ranked by
// counting, 512 at a time against all rows of the read passing through shared memory in tiles of 512.
__global__ void __launch_bounds__(512) rank_rows_big_kernel(uint32_t nreads, const uint64_t* __restrict__ read_coords, const uint32_t* __restrict__ slot,
                                                             const int4* __restrict__ k4, const uint32_t* __restrict__ k5,
                                                             uint32_t warp_max, uint32_t sort_cap, uint32_t* __restrict__ order) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const uint32_t r = blockIdx.x;
  if(r >= nreads) return;
  const uint64_t b = read_coords[r];
  const uint32_t c = (uint32_t)(read_coords[r + 1] - b);
  if(c <= warp_max) return;
  if(c <= sort_cap) {
    int4* s4 = (int4*)dyn;
    uint32_t* s5 = (uint32_t*)(s4 + sort_cap);
    uint32_t* idx = s5 + sort_cap;
    uint32_t m = 1;
    while(m < c) m <<= 1;
    for(uint32_t i = threadIdx.x; i < m; i += 512) {
      if(i < c) { s4[i] = k4[b + i]; s5[i] = k5[b + i]; idx[i] = i; }
      else idx[i] = prim::kPad;
    }
    __syncthreads();
    prim::bitonic_sort_idx(idx, (int)m, [&](uint32_t x, uint32_t y) {
      const int4 x4 = s4[x], y4 = s4[y];
      const row_key kx = { x4.x, x4.y, (uint32_t)x4.z, (uint32_t)x4.w, s5[x] }, ky = { y4.x, y4.y, (uint32_t)y4.z, (uint32_t)y4.w, s5[y] };
      if(row_key_less(kx, ky)) return true;
      if(row_key_less(ky, kx)) return false;
      return x < y;
    });
    for(uint32_t rk = threadIdx.x; rk < c; rk += 512) order[b + rk] = slot[b + idx[rk]];
    return;
  }
  int4* s4 = (int4*)dyn;                               // at least 512 entries of each (the launch sizes it)
  uint32_t* s5 = (uint32_t*)(s4 + 512);
  for(uint32_t e0 = 0; e0 < c; e0 += 512) {
    const uint32_t e = e0 + threadIdx.x;
    const bool mine = e < c;
    const int4 a4 = mine ? k4[b + e] : make_int4(0, 0, 0, 0);
    const row_key a = { a4.x, a4.y, (uint32_t)a4.z, (uint32_t)a4.w, mine ? k5[b + e] : 0u };
    uint32_t rank = 0;
    for(uint32_t f0 = 0; f0 < c; f0 += 512) {
      __syncthreads();
      if(f0 + threadIdx.x < c) { s4[threadIdx.x] = k4[b + f0 + threadIdx.x]; s5[threadIdx.x] = k5[b + f0 + threadIdx.x]; }
      __syncthreads();
      const uint32_t mm = min(512u, c - f0);
#pragma unroll 4
      for(uint32_t f = 0; f < mm; ++f) {
        const int4 o4 = s4[f];
        const row_key o = { o4.x, o4.y, (uint32_t)o4.z, (uint32_t)o4.w, s5[f] };
        rank += row_key_less(o, a);
      }
    }
    if(mine) order[b + rank] = slot[b + e];
  }
}

// largest number of coords rows any read of the batch has: the host picks the overlap-graph and
// row-ordering kernels with it
__global__ void __launch_bounds__(256) max_rows_kernel(const uint32_t* __restrict__ read_cnt, uint32_t nreads, unsigned long long* __restrict__ out) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t v = r < nreads ? read_cnt[r] : 0u;
  v = __reduce_max_sync(MR_FULL_MASK, v);
  if((threadIdx.x & 31) == 0 && v) atomicMax(out, (unsigned long long)v);
}

struct gather_args {
  uint64_t n; const uint32_t* order;
  survivors sv; const uint64_t* sv_info_off;
  coords_soa out;
};
__global__ void __launch_bounds__(256) gather_rows_kernel(gather_args A) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= A.n) return;
  const uint32_t s = A.order[i];
  A.out.rs[i] = A.sv.rs[s]; A.out.re[i] = A.sv.re[s]; A.out.qs[i] = A.sv.qs[s]; A.out.qe[i] = A.sv.qe[s];
  A.out.nb_mers[i] = A.sv.nb_mers[s];
  A.out.pb_cons[i] = A.sv.pb_cons[s]; A.out.sr_cons[i] = A.sv.sr_cons[s];
  A.out.pb_cover[i] = A.sv.pb_cover[s]; A.out.sr_cover[i] = A.sv.sr_cover[s];
  A.out.ql[i] = A.sv.ql[s]; A.out.sr[i] = A.sv.sr[s]; A.out.read[i] = A.sv.read[s];
  A.out.rn[i] = A.sv.rn[s]; A.out.use_bwd[i] = A.sv.use_bwd[s];
  A.out.stretch[i] = A.sv.stretch[s]; A.out.offset[i] = A.sv.offset[s]; A.out.avg_err[i] = A.sv.avg_err[s];
  A.out.info_off[i] = A.sv_info_off[s]; A.out.info_len[i] = A.sv.info_len[s];
  A.out.chain_pos[i] = A.sv.chain_pos[s];
}

// carve typed arrays out of one device buffer
template<typename T>
T* carve(char*& cursor, uint64_t count) {
  T* p = reinterpret_cast<T*>(cursor);
  cursor += ((count * sizeof(T) + 255) / 256) * 256;
  return p;
}

} // namespace

void mr_workspace_free(mr_workspace* ws) { delete ws; }

// ================================================================================================
// host orchestration
// L2 persistence window over the lookup tables of one index part for the kernels launched next on
// `st` (on == false: back to normal).  The tables (prefix counts + tails, index.cuh) are what every
// lookup reads at random; the 20 bytes per base the seed kernel streams out would otherwise keep
// evicting them (ncu: 40 % L2 hit rate with tables of 103 MB in a 126 MB L2).
static void l2_window(mr_context* ctx, cudaStream_t st, const mr_index* part, bool on) {
  if(!ctx->l2_persist_bytes || !part->lut.p) return;
  cudaStreamAttrValue v;
  memset(&v, 0, sizeof(v));
  if(on) {
    const size_t bytes = std::min(part->lut_bytes, ctx->l2_window_max);
    v.accessPolicyWindow.base_ptr = part->lut.p;
    v.accessPolicyWindow.num_bytes = bytes;
    v.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)ctx->l2_persist_bytes / (double)bytes);
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  }
  if(cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) cudaGetLastError();
}

// ================================================================================================
static int align_batch_impl(mr_context* ctx, mr_index* idx, const mr_params* p, const packed_reads& d_bases,
                            const uint64_t* d_read_start, const uint64_t* h_read_start, uint32_t nreads,
                            phase_timer& timer, mr_result** out) {
  cudaStream_t st = ctx->stream;
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  ws.graph_stamp = ws.rows_stamp = 0;      // the rows of the previous result are overwritten from here on
  const index_view& iv = idx->view;
  const uint32_t k = iv.k;
  const uint64_t T = h_read_start[nreads];
  if(T >= (1ULL << 32)) return ctx->fail(MR_ELIMIT, "mr_align_batch: more than 2^32 bases in one batch");
  if(nreads >= (1u << 31)) return ctx->fail(MR_ELIMIT, "mr_align_batch: too many reads in one batch");

  std::unique_ptr<mr_result> res(new mr_result);
  res->ctx = ctx;
  memset(&res->view, 0, sizeof(res->view));
  res->view.nreads = nreads;

  // ---- tiles (host side: O(#tiles)) ---------------------------------------------------------
  std::vector<uint32_t> tile_first(nreads + 1), tile_read, tile_pos, read_len(nreads);
  {
    uint64_t nt = 0;
    for(uint32_t r = 0; r < nreads; ++r) {
      const uint64_t len = h_read_start[r + 1] - h_read_start[r];
      if(len >= (1ULL << 31)) return ctx->fail(MR_ELIMIT, "mr_align_batch: read longer than 2^31 bases");
      read_len[r] = (uint32_t)len;
      tile_first[r] = (uint32_t)nt;
      nt += (len + kTile - 1) / kTile;
    }
    tile_first[nreads] = (uint32_t)nt;
    tile_read.resize(nt); tile_pos.resize(nt);
    for(uint32_t r = 0; r < nreads; ++r)
      for(uint32_t t = tile_first[r]; t < tile_first[r + 1]; ++t) { tile_read[t] = r; tile_pos[t] = (t - tile_first[r]) * kTile; }
  }
  const uint32_t ntiles = tile_first[nreads];
  MR_TRY(ws.tile_first.ensure(ctx, ((size_t)nreads + 1) * 4));
  MR_TRY(ws.read_len.ensure(ctx, ((size_t)nreads + 1) * 4));
  MR_TRY(ws.tile_read.ensure(ctx, ((size_t)ntiles + 1) * 4));
  MR_TRY(ws.tile_pos.ensure(ctx, ((size_t)ntiles + 1) * 4));
  MR_TRY(ws.tile_cand.ensure(ctx, ((size_t)ntiles + 1) * 4));
  MR_TRY(ws.tile_tbase.ensure(ctx, ((size_t)ntiles + 1) * 4));
  MR_TRY(ws.counters.ensure(ctx, 16 * sizeof(uint64_t)));
  MR_TRY(ws.size.ensure(ctx, (T + 4) * 4));
  const uint32_t nparts = idx->nparts();
  const uint64_t rec_stride = T + 4;
  MR_TRY(ws.rec.ensure(ctx, rec_stride * 16 * nparts));
  MR_TRY(ws.hit_off.ensure(ctx, ((size_t)ntiles + 4) * 8));
  MR_TRY(ws.thr.ensure(ctx, ((size_t)nreads + 1) * 4));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.tile_first.p, tile_first.data(), ((size_t)nreads + 1) * 4, cudaMemcpyHostToDevice, st));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.read_len.p, read_len.data(), (size_t)nreads * 4, cudaMemcpyHostToDevice, st));
  if(ntiles) {
    MR_CUDA(ctx, cudaMemcpyAsync(ws.tile_read.p, tile_read.data(), (size_t)ntiles * 4, cudaMemcpyHostToDevice, st));
    MR_CUDA(ctx, cudaMemcpyAsync(ws.tile_pos.p, tile_pos.data(), (size_t)ntiles * 4, cudaMemcpyHostToDevice, st));
  }
  MR_CUDA(ctx, cudaMemsetAsync(ws.counters.p, 0, 16 * sizeof(uint64_t), st));
  unsigned long long* ctr = ws.counters.as<unsigned long long>();
  // counters: 0 lookups, 1 raw hits, 2 invalid hits, 3 groups, 4 survivors, 5 info total, 6 tails, 7 fine hits,
  // 9 lists, 10 buckets, 11 tile overflow, 12 most rows of a read, 14 groups of hits that belong to no super-read
  uint64_t h_ctr[16] = { 0 };

  // ---- seeds + lookups ----------------------------------------------------------------------------
  timer.begin("seed prepass");
  if(ntiles) {
    MR_CUDA(ctx, cudaMemsetAsync(ws.tile_tbase.p, 0, (size_t)ntiles * 4, st));
    if(k <= 17) {
      seed_count_kernel<<<ntiles, kSeedThreads, 0, st>>>(d_bases, d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                       k, ws.tile_cand.as<uint32_t>());
      MR_LAUNCHED(ctx);
      tile_tbase_kernel<<<div_up(nreads, 128), 128, 0, st>>>(ws.tile_first.as<uint32_t>(), nreads, ws.tile_cand.as<uint32_t>(),
                                                             ws.tile_tbase.as<uint32_t>());
      MR_LAUNCHED(ctx);
    }
    timer.next("seed lookup");
    typedef void (*seed_fn)(index_view, uint32_t, packed_reads, const uint64_t*, const uint32_t*, const uint32_t*, const uint32_t*, uint32_t,
                            uint4*, uint32_t*, unsigned long long*, unsigned long long*, unsigned long long*, unsigned long long*);
    auto pick = [](bool multi, const index_view& v) -> seed_fn {
      const bool nibs = v.nib != nullptr, bytes = v.tail_bytes == 1;
      if(multi) return nibs ? (bytes ? seed_lookup_kernel<true, true, true> : seed_lookup_kernel<true, true, false>)
                            : (bytes ? seed_lookup_kernel<true, false, true> : seed_lookup_kernel<true, false, false>);
      return nibs ? (bytes ? seed_lookup_kernel<false, true, true> : seed_lookup_kernel<false, true, false>)
                  : (bytes ? seed_lookup_kernel<false, false, true> : seed_lookup_kernel<false, false, false>);
    };
    for(uint32_t part = 0; part < nparts; ++part) {
      l2_window(ctx, st, part ? idx->more[part - 1] : idx, true);
      const index_view& pv = idx->part_view(part);
      pick(nparts > 1, pv)<<<ntiles, kSeedThreads, 0, st>>>(pv, nparts == 1 ? 3u : ((part == 0 ? 1u : 0u) | (part + 1 == nparts ? 2u : 0u)),
                                                           d_bases, d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                           ws.tile_tbase.as<uint32_t>(), p->max_count > 0 ? (uint32_t)p->max_count : 0u,
                                                           ws.rec.as<uint4>() + part * rec_stride, ws.size.as<uint32_t>(), ctr + 0, ctr + 6, ctr + 9, ctr + 10);
      MR_LAUNCHED(ctx);
    }
    l2_window(ctx, st, idx, false);
    timer.next("count threshold");
    uint32_t nbits = 32;
    if(p->max_count > 1) { nbits = 0; while((1u << nbits) < (uint32_t)p->max_count) ++nbits; }
    else if(p->max_count == 1) nbits = 1;
    read_threshold_kernel<<<nreads, 256, 0, st>>>(d_read_start, nbits, ws.size.as<uint32_t>(), ws.thr.as<uint32_t>());
    MR_LAUNCHED(ctx);
  }
  timer.next("hit expansion");
  if(ntiles) {
    tile_hits_kernel<<<ntiles, kSeedThreads, 0, st>>>(d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                     ws.size.as<uint32_t>(), ws.tile_cand.as<uint32_t>(), ctr + 11);
    MR_LAUNCHED(ctx);
  }
  // tile_off[t] = first hit slot of tile t, tile_off[ntiles] = number of hits (also in counter 1)
  MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ ws.tile_cand.as<uint32_t>() }, ntiles, ws.hit_off.as<uint64_t>(),
                                                           ws.scan_scratch, (uint64_t*)(ctr + 1))));
  if(ntiles) MR_CUDA(ctx, cudaMemcpyAsync(ws.hit_off.as<uint64_t>() + ntiles, ctr + 1, sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
  int sr_bits = 1;
  while((1ULL << sr_bits) <= (uint64_t)iv.nseq_all) ++sr_bits;
  MR_CUDA(ctx, cudaMemcpyAsync(h_ctr, ctr, 12 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  MR_CUDA(ctx, ctx->wait(st));
  if(h_ctr[11]) return ctx->fail(MR_ELIMIT, "mr_align_batch: 2^32 or more hits in one 1024-base tile; use --max-count");
  const uint64_t H = h_ctr[1];
  MR_TRACE_MSG("batch: %u reads, %llu bases, %llu lookups, %llu raw hits", nreads, (unsigned long long)T, (unsigned long long)h_ctr[0], (unsigned long long)H);
  res->view.n_kmers_looked_up = h_ctr[0];
  res->view.n_tail_entries = h_ctr[6];
  res->view.n_lists = h_ctr[9];
  res->view.n_buckets = h_ctr[10];
  // MR_MAX_HITS lowers the limit (tests of the callers' batch splitting)
  static const uint64_t hit_limit = getenv("MR_MAX_HITS") ? strtoull(getenv("MR_MAX_HITS"), nullptr, 0) : (1ULL << 32);
  if(H >= hit_limit) return ctx->fail(MR_ELIMIT, "mr_align_batch: too many hits in one batch; use smaller batches");

  uint64_t G = 0, S = 0, cap = 0;
  const bool taps = ctx->keep_taps;
  uint64_t *skeys = nullptr, *spays = nullptr;
  chain_args A;
  memset(&A, 0, sizeof(A));
  if(H) {
    MR_TRY(ws.key0.ensure(ctx, (H + 2) * 8)); MR_TRY(ws.key1.ensure(ctx, (H + 2) * 8));
    MR_TRY(ws.pay0.ensure(ctx, (H + 2) * 8)); MR_TRY(ws.pay1.ensure(ctx, (H + 2) * 8));
    if(nparts == 1)
      expand_kernel<false><<<ntiles, kSeedThreads, 0, st>>>(iv, nullptr, 1, 0, d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                          ws.rec.as<uint4>(), ws.size.as<uint32_t>(), ws.hit_off.as<uint64_t>(),
                                                          ws.key0.as<uint64_t>(), ws.pay0.as<uint64_t>(), ctr + 2);
    else
      expand_kernel<true><<<ntiles, kSeedThreads, 0, st>>>(iv, idx->more_views.as<index_view>(), nparts, rec_stride, d_read_start,
                                                         ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                         ws.rec.as<uint4>(), ws.size.as<uint32_t>(), ws.hit_off.as<uint64_t>(),
                                                         ws.key0.as<uint64_t>(), ws.pay0.as<uint64_t>(), ctr + 2);
    MR_LAUNCHED(ctx);
    timer.next("group sort");
    // Grouping by (read, super-read): one CTA per read (group.cu), in shared memory when the read's hits fit,
    // through one cut by the top bits of the super-read index when they do not.  An index of more than 2^25
    // super-reads, or MR_READ_SORT=0, takes the device-wide radix sort instead.
    static const bool read_sort_on = !(getenv("MR_READ_SORT") && atoi(getenv("MR_READ_SORT")) == 0);
    const bool read_sort = read_sort_on && group_sort_usable(sr_bits);
    uint64_t *alt_key, *alt_pay;
    if(read_sort) {
      MR_TRY(ws.head.ensure(ctx, H + 2));
      group_sort_args GS;
      GS.keys_in = ws.key0.as<uint64_t>(); GS.pays_in = ws.pay0.as<uint64_t>();
      GS.keys_out = ws.key1.as<uint64_t>(); GS.pays_out = ws.pay1.as<uint64_t>();
      GS.head = ws.head.as<uint8_t>(); GS.hit_off = ws.hit_off.as<uint64_t>(); GS.tile_first = ws.tile_first.as<uint32_t>();
      GS.nseq_all = iv.nseq_all; GS.sr_bits = sr_bits; GS.n_invalid_groups = ctr + 14; GS.cap = 0; GS.idx_bits = 0;
      MR_TRY(launch_group_sort(ctx, GS, nreads));
      skeys = GS.keys_out; spays = GS.pays_out; alt_key = GS.keys_in; alt_pay = GS.pays_in;
      MR_TRY((prim::flag_count<head_byte>(ctx, head_byte{ GS.head }, H, ws.scan_scratch, (uint64_t*)(ctr + 3))));
    } else {
      bool in_first = true;
      MR_TRY((prim::radix_sort_pairs<uint64_t, uint64_t>(ctx, ws.key0.as<uint64_t>(), ws.pay0.as<uint64_t>(), ws.key1.as<uint64_t>(),
                                                         ws.pay1.as<uint64_t>(), H, 0, sr_bits, ws.sort, &in_first)));
      skeys = in_first ? ws.key0.as<uint64_t>() : ws.key1.as<uint64_t>();
      spays = in_first ? ws.pay0.as<uint64_t>() : ws.pay1.as<uint64_t>();
      alt_key = in_first ? ws.key1.as<uint64_t>() : ws.key0.as<uint64_t>();
      alt_pay = in_first ? ws.pay1.as<uint64_t>() : ws.pay0.as<uint64_t>();
      // group heads -> group_start
      MR_TRY((prim::flag_count<head_flag>(ctx, head_flag{ skeys, iv.nseq_all }, H, ws.scan_scratch, (uint64_t*)(ctr + 3))));
    }
    MR_CUDA(ctx, cudaMemcpyAsync(h_ctr, ctr, 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
    G = h_ctr[3];
    MR_TRACE_MSG("sorted (%s); %llu groups", read_sort ? "per read" : "device-wide", (unsigned long long)G);
    const uint64_t Hvalid = H - h_ctr[2];
    res->view.n_hits = Hvalid;
    res->view.n_groups = G - (read_sort ? h_ctr[14] : 0);      // (the per-read sort makes a group of a read's stray hits)
    MR_TRY(ws.group_start.ensure(ctx, (G + 2) * 8));
    if(read_sort) {
      MR_TRY((prim::flag_positions<head_byte>(ctx, head_byte{ ws.head.as<uint8_t>() }, H, ws.scan_scratch, ws.group_start.as<uint64_t>())));
      // the stray hits stay inside their reads' slices: the last group ends with the last hit
      MR_CUDA(ctx, cudaMemcpyAsync(ws.group_start.as<uint64_t>() + G, ctr + 1, 8, cudaMemcpyDeviceToDevice, st));
    } else {
      MR_TRY((prim::flag_positions<head_flag>(ctx, head_flag{ skeys, iv.nseq_all }, H, ws.scan_scratch, ws.group_start.as<uint64_t>())));
      // end of the last group; the source lives in the result object (a copy from pageable memory is staged before the call returns)
      MR_CUDA(ctx, cudaMemcpyAsync(ws.group_start.as<uint64_t>() + G, &res->view.n_hits, 8, cudaMemcpyHostToDevice, st));
    }

    // ---- chaining + coords ------------------------------------------------------------------------
    timer.next("chain coords");
    MR_TRY(ws.chainL.ensure(ctx, (H + 2) * 16));
    MR_TRY(ws.read_cnt.ensure(ctx, ((size_t)nreads + 2) * 4));
    A.iv = iv; A.sr_len = idx->sr_len.as<uint32_t>(); A.keys = skeys; A.pays = spays; A.group_start = ws.group_start.as<uint64_t>(); A.ngroups = G;
    A.read_start = d_read_start;
    {
      char* c = (char*)ws.chainL.p;
      A.cb.Lpb = (int32_t*)c; A.cb.Lsr = (int32_t*)(c + (H + 2) * 4); A.cb.Llen = (uint32_t*)(c + (H + 2) * 8);
      A.cb.Lelt = (uint32_t*)(c + (H + 2) * 12);
      A.cb.pprev = (uint32_t*)alt_pay; A.cb.cstart = (uint32_t*)alt_pay + (H + 2);
    }
    A.window = p->window_size;
    if(p->window_size > 1) {
      MR_TRY(ws.chainW.ensure(ctx, (H + 2) * 8));
      A.cb.Lwpb = ws.chainW.as<int32_t>(); A.cb.Lwsr = ws.chainW.as<int32_t>() + (H + 2);
    }
    A.a = p->stretch_factor; A.b = p->stretch_constant; A.C = p->stretch_cap;
    A.matching_mers = p->matching_mers; A.matching_bases = p->matching_bases; A.forward = p->forward;
    A.unitigs_k = idx->has_unitigs ? p->unitigs_k : 0; A.n_unitigs = idx->n_unitigs;
    A.unitig_ids = idx->unitig_ids.as<uint32_t>(); A.unitig_off = idx->has_unitigs ? idx->unitig_off.as<uint64_t>() : nullptr;
    A.chain_pay = alt_key;                  // gpos is dead once group_start exists
    if(taps) {
      MR_TRY(ws.chain_pay.ensure(ctx, (H + 2) * 8));
      A.chain_pay = ws.chain_pay.as<uint64_t>();   // with taps on, alt_key holds the sub-list indices instead
      MR_TRY(ws.tap_lens.ensure(ctx, (G + 1) * 8));
      MR_TRY(ws.tap_cf.ensure(ctx, (H + 2) * 4)); MR_TRY(ws.tap_cb.ensure(ctx, (H + 2) * 4));
      A.tap_lens = ws.tap_lens.as<uint2>(); A.tap_cf = ws.tap_cf.as<uint32_t>(); A.tap_cb = ws.tap_cb.as<uint32_t>();
      A.tap_sub = (uint32_t*)alt_key;       // gpos is dead once group_start exists
    }
    cap = std::max<uint64_t>(1 << 20, G / 4 + 1024);
    if(cap > G && !p->max_match) cap = G;
    if(cap == 0) cap = 1;
    A.max_match = p->max_match;
    if(p->max_match) { MR_TRY(ws.removed.ensure(ctx, H + 2)); A.removed = ws.removed.as<uint8_t>(); }
    for(int attempt = 0; attempt < 2; ++attempt) {
      MR_TRY(ws.sv_i32.ensure(ctx, cap * 4 * 5 + 4096)); MR_TRY(ws.sv_u32.ensure(ctx, cap * 4 * 9 + 4096));
      MR_TRY(ws.sv_f64.ensure(ctx, cap * 8 * 3 + 4096)); MR_TRY(ws.sv_u64.ensure(ctx, cap * 8 * 2 + 4096));
      MR_TRY(ws.sv_u8.ensure(ctx, cap * 2 + 4096));
      survivors& sv = A.sv;
      { int32_t* b = ws.sv_i32.as<int32_t>(); sv.rs = b; sv.re = b + cap; sv.qs = b + 2 * cap; sv.qe = b + 3 * cap; sv.nb_mers = b + 4 * cap; }
      { uint32_t* b = ws.sv_u32.as<uint32_t>(); sv.pb_cons = b; sv.sr_cons = b + cap; sv.pb_cover = b + 2 * cap; sv.sr_cover = b + 3 * cap;
        sv.ql = b + 4 * cap; sv.sr = b + 5 * cap; sv.read = b + 6 * cap; sv.info_len = b + 7 * cap; sv.iter = b + 8 * cap; }
      { double* b = ws.sv_f64.as<double>(); sv.stretch = b; sv.offset = b + cap; sv.avg_err = b + 2 * cap; }
      { uint64_t* b = ws.sv_u64.as<uint64_t>(); sv.chain_pos = b; }
      { uint8_t* b = ws.sv_u8.as<uint8_t>(); sv.rn = b; sv.use_bwd = b + cap; }
      sv.cap = cap; sv.count = ctr + 4; sv.info_total = ctr + 5; sv.read_cnt = ws.read_cnt.as<uint32_t>();
      MR_CUDA(ctx, cudaMemsetAsync(ctr + 4, 0, 2 * sizeof(uint64_t), st));
      MR_CUDA(ctx, cudaMemsetAsync(ws.read_cnt.p, 0, ((size_t)nreads + 2) * 4, st));
      if(G) MR_TRY(launch_chain(ctx, A, ws.group_lists));
      max_rows_kernel<<<div_up(nreads, 256), 256, 0, st>>>(ws.read_cnt.as<uint32_t>(), nreads, ctr + 12);
      MR_LAUNCHED(ctx);
      MR_CUDA(ctx, cudaMemcpyAsync(h_ctr, ctr, 13 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
      MR_CUDA(ctx, ctx->wait(st));
      S = h_ctr[4];
      MR_TRACE_MSG("chained; %llu rows (capacity %llu)", (unsigned long long)S, (unsigned long long)cap);
      if(S <= cap) break;
      cap = S;                                 // rare: more survivors than provisioned, run again
    }
  } else {
    MR_TRY(ws.read_cnt.ensure(ctx, ((size_t)nreads + 2) * 4));
    MR_CUDA(ctx, cudaMemsetAsync(ws.read_cnt.p, 0, ((size_t)nreads + 2) * 4, st));
  }
  if(S >= (1ULL << 32)) return ctx->fail(MR_ELIMIT, "mr_align_batch: more than 2^32 coords rows");
  uint32_t k_coords = k;                                 // mer length of the rows that go on (kmers_info)

  // ---- fine pass (-F): the coarse rows become windows, their coords are recomputed from shorter mers -----
  if(p->fine_mer && S) {
    timer.next("fine pass");
    const uint32_t kk = p->fine_mer;
    fine_buffers& fb = ws.fine;
    MR_TRY(fb.wkey0.ensure(ctx, S * 8)); MR_TRY(fb.wkey1.ensure(ctx, S * 8)); MR_TRY(fb.wrow0.ensure(ctx, S * 4)); MR_TRY(fb.wrow1.ensure(ctx, S * 4));
    MR_TRY(fb.wbegin.ensure(ctx, S * 8)); MR_TRY(fb.wend.ensure(ctx, S * 8));
    MR_TRY(fb.gread.ensure(ctx, S * 4)); MR_TRY(fb.gsr.ensure(ctx, S * 4)); MR_TRY(fb.giter.ensure(ctx, S * 4));
    MR_TRY(fb.table_off.ensure(ctx, ((size_t)nreads + 2) * 8));
    MR_TRY(fb.row_cnt.ensure(ctx, (S + 2) * 4)); MR_TRY(fb.group_start.ensure(ctx, (S + 2) * 8));
    // rows of read r in the (read, super-read)-sorted table: [table_off[r], table_off[r + 1])
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ ws.read_cnt.as<uint32_t>() }, (uint64_t)nreads + 1,
                                                             fb.table_off.as<uint64_t>(), ws.scan_scratch, nullptr)));
    fine_windows_kernel<<<div_up(S, 256), 256, 0, st>>>(S, A.sv, d_read_start, kk, fb.wkey0.as<uint64_t>(), fb.wrow0.as<uint32_t>(),
                                                        fb.wbegin.as<double>(), fb.wend.as<double>(), fb.gread.as<uint32_t>(),
                                                        fb.gsr.as<uint32_t>(), fb.giter.as<uint32_t>());
    MR_LAUNCHED(ctx);
    int sr_bits = 1, read_bits = 1;
    while((1ULL << sr_bits) <= (uint64_t)iv.nseq_all) ++sr_bits;
    while((1ULL << read_bits) <= (uint64_t)nreads) ++read_bits;
    bool first = true;
    MR_TRY((prim::radix_sort_pairs<uint64_t, uint32_t>(ctx, fb.wkey0.as<uint64_t>(), fb.wrow0.as<uint32_t>(), fb.wkey1.as<uint64_t>(),
                                                       fb.wrow1.as<uint32_t>(), S, 0, sr_bits, fb.sort, &first)));
    uint64_t *wk_a = first ? fb.wkey0.as<uint64_t>() : fb.wkey1.as<uint64_t>(), *wk_b = first ? fb.wkey1.as<uint64_t>() : fb.wkey0.as<uint64_t>();
    uint32_t *wr_a = first ? fb.wrow0.as<uint32_t>() : fb.wrow1.as<uint32_t>(), *wr_b = first ? fb.wrow1.as<uint32_t>() : fb.wrow0.as<uint32_t>();
    MR_TRY((prim::radix_sort_pairs<uint64_t, uint32_t>(ctx, wk_a, wr_a, wk_b, wr_b, S, 32, 32 + read_bits, fb.sort, &first)));
    const uint64_t* tkey = first ? wk_a : wk_b;
    const uint32_t* trow = first ? wr_a : wr_b;
    if(ntiles) {
      for(uint32_t part = 0; part < nparts; ++part) {
        fine_seed_kernel<<<ntiles, kSeedThreads, 0, st>>>(idx->part_view(part), part == 0, kk, d_bases, d_read_start, ws.tile_read.as<uint32_t>(),
                                                          ws.tile_pos.as<uint32_t>(), fb.table_off.as<uint64_t>(),
                                                          ws.rec.as<uint4>() + part * rec_stride, ws.size.as<uint32_t>());
        MR_LAUNCHED(ctx);
      }
    }
    MR_CUDA(ctx, cudaMemsetAsync(fb.row_cnt.p, 0, (S + 2) * 4, st));
    fine_expand_kernel<false><<<ntiles, kSeedThreads, 0, st>>>(iv, idx->more_views.as<index_view>(), nparts, rec_stride, kk, d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                             ws.rec.as<uint4>(), ws.size.as<uint32_t>(), fb.table_off.as<uint64_t>(), tkey, trow,
                                                             fb.wbegin.as<double>(), fb.wend.as<double>(), ws.tile_cand.as<uint32_t>(), nullptr,
                                                             fb.row_cnt.as<uint32_t>(), nullptr, nullptr);
    MR_LAUNCHED(ctx);
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ ws.tile_cand.as<uint32_t>() }, ntiles, ws.hit_off.as<uint64_t>(),
                                                             ws.scan_scratch, (uint64_t*)(ctr + 7))));
    MR_CUDA(ctx, cudaMemcpyAsync(ws.hit_off.as<uint64_t>() + ntiles, ctr + 7, sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    MR_CUDA(ctx, cudaMemcpyAsync(h_ctr + 7, ctr + 7, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
    const uint64_t Hf = h_ctr[7];
    MR_TRACE_MSG("fine pass: %llu windows, %llu hits inside them", (unsigned long long)S, (unsigned long long)Hf);
    if(Hf >= (1ULL << 32)) return ctx->fail(MR_ELIMIT, "mr_align_batch: too many fine-pass hits in one batch; use smaller batches");
    MR_TRY(ws.key0.ensure(ctx, (Hf + 2) * 8)); MR_TRY(ws.key1.ensure(ctx, (Hf + 2) * 8));
    MR_TRY(ws.pay0.ensure(ctx, (Hf + 2) * 8)); MR_TRY(ws.pay1.ensure(ctx, (Hf + 2) * 8));
    MR_TRY(ws.chainL.ensure(ctx, (Hf + 2) * 16));
    if(Hf) {
      fine_expand_kernel<true><<<ntiles, kSeedThreads, 0, st>>>(iv, idx->more_views.as<index_view>(), nparts, rec_stride, kk, d_read_start, ws.tile_read.as<uint32_t>(), ws.tile_pos.as<uint32_t>(),
                                                              ws.rec.as<uint4>(), ws.size.as<uint32_t>(), fb.table_off.as<uint64_t>(), tkey, trow,
                                                              fb.wbegin.as<double>(), fb.wend.as<double>(), nullptr, ws.hit_off.as<uint64_t>(),
                                                              nullptr, ws.key0.as<uint64_t>(), ws.pay0.as<uint64_t>());
      MR_LAUNCHED(ctx);
    }
    int row_bits = 1;
    while((1ULL << row_bits) < S) ++row_bits;
    bool in_first = true;
    MR_TRY((prim::radix_sort_pairs<uint64_t, uint64_t>(ctx, ws.key0.as<uint64_t>(), ws.pay0.as<uint64_t>(), ws.key1.as<uint64_t>(),
                                                       ws.pay1.as<uint64_t>(), Hf, 0, row_bits, ws.sort, &in_first)));
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ fb.row_cnt.as<uint32_t>() }, S + 1,
                                                             fb.group_start.as<uint64_t>(), ws.scan_scratch, nullptr)));
    chain_args F = A;
    F.keys = in_first ? ws.key0.as<uint64_t>() : ws.key1.as<uint64_t>();
    F.pays = in_first ? ws.pay0.as<uint64_t>() : ws.pay1.as<uint64_t>();
    uint64_t* f_alt_key = in_first ? ws.key1.as<uint64_t>() : ws.key0.as<uint64_t>();
    uint64_t* f_alt_pay = in_first ? ws.pay1.as<uint64_t>() : ws.pay0.as<uint64_t>();
    F.group_start = fb.group_start.as<uint64_t>(); F.ngroups = S;
    {
      char* cb = (char*)ws.chainL.p;
      F.cb.Lpb = (int32_t*)cb; F.cb.Lsr = (int32_t*)(cb + (Hf + 2) * 4); F.cb.Llen = (uint32_t*)(cb + (Hf + 2) * 8);
      F.cb.Lelt = (uint32_t*)(cb + (Hf + 2) * 12);
      F.cb.pprev = (uint32_t*)f_alt_pay; F.cb.cstart = (uint32_t*)f_alt_pay + (Hf + 2);
    }
    F.chain_pay = f_alt_key;
    F.a = -1.0; F.b = 0.0; F.C = -1.0;                    // lis_align::accept_all
    F.matching_mers = 0.0; F.matching_bases = 0.0; F.forward = 1; F.no_filter = 1; F.align_k = kk;
    F.group_read = fb.gread.as<uint32_t>(); F.group_sr = fb.gsr.as<uint32_t>(); F.group_iter = fb.giter.as<uint32_t>();
    F.max_match = 0; F.removed = nullptr; F.window = 1;            // accept-all predicates: a window changes nothing
    F.tap_lens = nullptr; F.tap_cf = nullptr; F.tap_cb = nullptr; F.tap_sub = nullptr;
    MR_CUDA(ctx, cudaMemsetAsync(ctr + 4, 0, 2 * sizeof(uint64_t), st));
    MR_CUDA(ctx, cudaMemsetAsync(ws.read_cnt.p, 0, ((size_t)nreads + 2) * 4, st));
    MR_TRY(launch_chain(ctx, F, ws.group_lists));
    MR_CUDA(ctx, cudaMemcpyAsync(h_ctr, ctr, 6 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
    if(h_ctr[4] != S) return ctx->fail(MR_ECUDA, "mr_align_batch: internal error, the fine pass lost rows");
    A = F;
    k_coords = kk;
  }
  const uint64_t info_total = S ? h_ctr[5] : 0;
  const int max_rows = S ? (int)std::min<uint64_t>(h_ctr[12], 0x7fffffff) : 0;      // rows of the read that has most

  // ---- kmers_info, per-read order, final rows ---------------------------------------------------
  timer.next("coords order");
  MR_TRY(ws.read_coords.ensure(ctx, ((size_t)nreads + 2) * 8));
  MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ ws.read_cnt.as<uint32_t>() }, (uint64_t)nreads + 1,
                                                           ws.read_coords.as<uint64_t>(), ws.scan_scratch, nullptr)));
  coords_soa fin;
  const uint64_t Sc = std::max<uint64_t>(S, 1);
  MR_TRY(setup_final_rows(ctx, ws, Sc, fin));
  uint64_t* sv_info_off = ws.fin_u64.as<uint64_t>() + 2 * Sc;
  MR_TRY(ws.kinfo.ensure(ctx, (info_total + 1) * 4)); MR_TRY(ws.binfo.ensure(ctx, (info_total + 1) * 4));
  if(S) {
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ A.sv.info_len }, S, sv_info_off, ws.scan_scratch, nullptr)));
    if(info_total) {
      info_args I;
      I.n = S; I.chain_pos = A.sv.chain_pos; I.nb_mers = A.sv.nb_mers; I.sr = A.sv.sr; I.use_bwd = A.sv.use_bwd; I.ql = A.sv.ql;
      I.info_off = sv_info_off; I.info_len = A.sv.info_len; I.chain_pay = A.chain_pay;
      I.unitig_ids = idx->unitig_ids.as<uint32_t>(); I.unitig_off = idx->unitig_off.as<uint64_t>();
      I.unitig_len = idx->unitig_len.as<int32_t>(); I.n_unitigs = idx->n_unitigs; I.k = k_coords; I.unitigs_k = p->unitigs_k;
      I.kinfo = ws.kinfo.as<int32_t>(); I.binfo = ws.binfo.as<int32_t>();
      kmers_info_kernel<<<div_up(S, 4), 128, 0, st>>>(I);
      MR_LAUNCHED(ctx);
    }
    MR_TRY(ws.read_cursor.ensure(ctx, ((size_t)nreads + 1) * 4));
    MR_TRY(ws.slot.ensure(ctx, S * 4)); MR_TRY(ws.order.ensure(ctx, S * 4));
    MR_CUDA(ctx, cudaMemsetAsync(ws.read_cursor.p, 0, ((size_t)nreads + 1) * 4, st));
    bucket_rows_kernel<<<div_up(S, 256), 256, 0, st>>>(S, A.sv.read, ws.read_coords.as<uint64_t>(), ws.read_cursor.as<uint32_t>(),
                                                       ws.slot.as<uint32_t>());
    MR_LAUNCHED(ctx);
    MR_TRY(ws.rowkey4.ensure(ctx, S * sizeof(int4))); MR_TRY(ws.rowkey5.ensure(ctx, S * sizeof(uint32_t)));
    row_keys_kernel<<<div_up(S, 256), 256, 0, st>>>(S, ws.slot.as<uint32_t>(), A.sv.rs, A.sv.re, A.sv.ql, A.sv.sr, A.sv.iter,
                                                    ws.rowkey4.as<int4>(), ws.rowkey5.as<uint32_t>());
    MR_LAUNCHED(ctx);
    rank_rows_kernel<<<div_up((uint64_t)nreads * 32, 128), 128, 0, st>>>(nreads, ws.read_coords.as<uint64_t>(), ws.slot.as<uint32_t>(),
                                                                                ws.rowkey4.as<int4>(), ws.rowkey5.as<uint32_t>(), (uint32_t)big_rows_threshold(), ws.order.as<uint32_t>());
    MR_LAUNCHED(ctx);
    if(max_rows > big_rows_threshold()) {                            // some read has that many rows
      uint32_t sort_cap = 512;
      while(sort_cap < (uint32_t)std::min(max_rows, big_sort_rows_limit())) sort_cap <<= 1;
      const size_t smem = (size_t)std::max<uint32_t>(sort_cap, 512) * 24;
      MR_CUDA(ctx, cudaFuncSetAttribute(rank_rows_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      rank_rows_big_kernel<<<nreads, 512, smem, st>>>(nreads, ws.read_coords.as<uint64_t>(), ws.slot.as<uint32_t>(),
                                                    ws.rowkey4.as<int4>(), ws.rowkey5.as<uint32_t>(), (uint32_t)big_rows_threshold(),
                                                    std::min<uint32_t>(sort_cap, (uint32_t)big_sort_rows_limit()), ws.order.as<uint32_t>());
      MR_LAUNCHED(ctx);
    }
    gather_args Gt;
    Gt.n = S; Gt.order = ws.order.as<uint32_t>(); Gt.sv = A.sv; Gt.sv_info_off = sv_info_off; Gt.out = fin;
    gather_rows_kernel<<<div_up(S, 256), 256, 0, st>>>(Gt);
    MR_LAUNCHED(ctx);
  }

  // ---- overlap graph -----------------------------------------------------------------------------
  const bool graph = p->run_graph != 0;
  graph_args GA;
  memset(&GA, 0, sizeof(GA));
  if(graph) {
    timer.next("overlap graph");
    GA.nreads = nreads; GA.read_coords = ws.read_coords.as<uint64_t>(); GA.read_len = ws.read_len.as<uint32_t>(); GA.c = fin;
    GA.kinfo = ws.kinfo.as<int32_t>(); GA.binfo = ws.binfo.as<int32_t>();
    GA.unitig_ids = idx->unitig_ids.as<uint32_t>(); GA.unitig_off = idx->has_unitigs ? idx->unitig_off.as<uint64_t>() : nullptr;
    GA.unitig_len = idx->unitig_len.as<int32_t>(); GA.n_unitigs = idx->n_unitigs; GA.unitigs_k = p->unitigs_k;
    GA.overlap_play = p->overlap_play; GA.errors = p->errors; GA.bases = p->bases; GA.warp_max_rows = big_rows_threshold();
    MR_TRY(setup_graph_nodes(ctx, ws, Sc, GA));
    if(S) MR_TRY(launch_graph(ctx, ws, GA, S, max_rows));
  }
  timer.next("result download");
  MR_TRACE_MSG("ordered%s; downloading", graph ? " + graph" : "");

  // ---- results to pinned host memory ----------------------------------------------------------------
  MR_TRY(download_rows(ctx, ws, res.get(), fin, nreads, S, info_total, graph ? &GA : nullptr));

  // ---- parity taps: (read, super-read) hit lists and both chains, rows sorted by (read, sr) ------
  // (--max-match: the lists after every discard, i.e. without the hits of the emitted chains that were removed)
  if(taps && G) {
    std::vector<uint64_t> hk(H), hp(H), hg(G + 1);
    std::vector<uint2> hl(G);
    std::vector<uint32_t> hcf(H), hcb(H);
    std::vector<uint8_t> hrem(p->max_match ? H : 0);
    MR_CUDA(ctx, cudaMemcpyAsync(hk.data(), skeys, H * 8, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, cudaMemcpyAsync(hp.data(), spays, H * 8, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, cudaMemcpyAsync(hg.data(), ws.group_start.p, (G + 1) * 8, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, cudaMemcpyAsync(hl.data(), ws.tap_lens.p, G * 8, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, cudaMemcpyAsync(hcf.data(), ws.tap_cf.p, H * 4, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, cudaMemcpyAsync(hcb.data(), ws.tap_cb.p, H * 4, cudaMemcpyDeviceToHost, st));
    if(p->max_match) MR_CUDA(ctx, cudaMemcpyAsync(hrem.data(), ws.removed.p, H, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
    auto kept = [&](uint64_t i) { return hrem.empty() || !hrem[i]; };
    std::vector<uint64_t> ord(G);
    for(uint64_t g = 0; g < G; ++g) ord[g] = g;
    std::sort(ord.begin(), ord.end(), [&](uint64_t a, uint64_t b) { return hk[hg[a]] < hk[hg[b]]; });
    for(uint64_t g : ord) {
      const uint64_t b = hg[g], e = hg[g + 1];
      if((uint32_t)hk[b] == iv.nseq_all) continue;        // a read's hits that belong to no super-read
      int64_t nf = 0, nbw = 0;
      for(uint64_t i = b; i < e; ++i) if(kept(i)) ((int32_t)(uint32_t)(hp[i] >> 32) > 0 ? nf : nbw)++;
      const int64_t row[6] = { (int64_t)(hk[b] >> 32), (int64_t)(uint32_t)hk[b], nf, nbw, hl[g].x, hl[g].y };
      res->tap_groups.insert(res->tap_groups.end(), row, row + 6);
      for(int pass = 0; pass < 2; ++pass)
        for(uint64_t i = b; i < e; ++i) {
          const int32_t so = (int32_t)(uint32_t)(hp[i] >> 32);
          if(kept(i) && (so > 0) == (pass == 0)) { res->tap_offsets.push_back((int32_t)(uint32_t)hp[i]); res->tap_offsets.push_back(so); }
        }
      for(uint32_t t = 0; t < hl[g].x; ++t) res->tap_lis.push_back(hcf[b + t]);
      for(uint32_t t = 0; t < hl[g].y; ++t) res->tap_lis.push_back(hcb[b + t]);
    }
  }
  timer.end();
  MR_CUDA(ctx, ctx->wait(st));
  MR_TRACE_MSG("batch done");
  remember_rows(ws, res.get(), fin, nreads, graph ? &GA : nullptr, S, max_rows);
  *out = res.release();
  return MR_OK;
}

// checks shared by every alignment entry point, then the batch itself on packed device arrays
static int align_checked(mr_context* ctx, mr_index* idx, const mr_params* p, const packed_reads& d_reads,
                         const uint64_t* d_read_start, const uint64_t* h_read_start, uint32_t nreads, mr_result** out) {
  if(!idx || !p || !out || !h_read_start || !d_read_start) return ctx->fail(MR_EINVAL, "mr_align_batch: null argument");
  // an index is read-only once built: any context of its device may align against it
  if(idx->ctx->device != ctx->device) return ctx->fail(MR_EINVAL, "mr_align_batch: index lives on another device");
  if(p->window_size < 1) return ctx->fail(MR_EINVAL, "mr_align_batch: --window-size must be at least 1");
  if(p->fine_mer && ctx->keep_taps) return ctx->fail(MR_EINVAL, "mr_align_batch: parity taps are not available with a fine pass");
  if(p->fine_mer && (p->fine_mer < idx->m || p->fine_mer > idx->k))
    return ctx->fail(MR_EINVAL, "mr_align_batch: the fine mer must lie between the psa_min and the mer length the index was built with "
                                "(the reference builds its suffix array with min(fine mer, psa-min), create_mega_reads.cc:131-132)");
  if(p->run_graph && !(idx->has_unitigs && p->unitigs_k))
    return ctx->fail(MR_EINVAL, "mr_align_batch: the overlap graph needs unitig lengths (-l/-u) and -k");
  if(p->run_graph && !idx->unitig_ids_ok)
    return ctx->fail(MR_EINVAL, "mr_align_batch: a super-read name refers to a k-unitig that the unitig table (-l/-u) does not have");
  ctx->timers.clear();
  phase_timer timer(ctx);
  const int rc = align_batch_impl(ctx, idx, p, d_reads, d_read_start, h_read_start, nreads, timer, out);
  cudaStreamSynchronize(ctx->stream);
  if(rc == MR_OK) timer.collect();
  else {
    // a failed batch may have left kernels of the chain tiers running on the side streams: the caller
    // retries with a smaller batch, which re-sizes the very buffers they use
    for(cudaStream_t s : ctx->aux) if(s) cudaStreamSynchronize(s);
    for(cudaStream_t s : ctx->hi) if(s) cudaStreamSynchronize(s);
    cudaGetLastError();
  }
  return rc;
}

static bool g_no_tma() { static const bool v = getenv("MR_NO_TMA") && atoi(getenv("MR_NO_TMA")) != 0; return v; }
static packed_reads make_packed(const uint64_t* codes, const uint64_t* nmask) {
  packed_reads r;
  r.codes = codes; r.nmask = nmask;
  r.tma = !g_no_tma() && (((uintptr_t)codes | (uintptr_t)nmask) & 15) == 0;
  return r;
}

// characters already on the device -> the context's packed buffers
static int pack_on_device(mr_context* ctx, const char* d_bases, uint64_t T, packed_reads& out) {
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  const uint64_t mwords = mr_packed_mask_words(T), cwords = mr_packed_code_words(T);
  MR_TRY(ws.codes.ensure(ctx, cwords * 8)); MR_TRY(ws.nmask.ensure(ctx, mwords * 8));
  // the kernel writes whole 64-base groups; the padding words behind them stay whatever they are (never decoded)
  const uint64_t groups = (T + 63) / 64;
  if(groups) {
    pack_reads_kernel<<<div_up(groups, 256), 256, 0, ctx->stream>>>(d_bases, T, ws.codes.as<uint64_t>(), ws.nmask.as<uint64_t>(), groups);
    MR_LAUNCHED(ctx);
  }
  out = make_packed(ws.codes.as<uint64_t>(), ws.nmask.as<uint64_t>());
  return MR_OK;
}

extern "C" {

// (mr_packed_code_words / mr_packed_mask_words / mr_pack_reads / mr_pack_reads_range: pack_host.cpp)

int mr_align_batch_device(mr_context* ctx, mr_index* idx, const mr_params* p, const char* d_bases,
                          const uint64_t* d_read_start, const uint64_t* h_read_start, uint32_t nreads, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!d_bases || !h_read_start) return ctx->fail(MR_EINVAL, "mr_align_batch: null argument");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  packed_reads pr;
  MR_TRY(pack_on_device(ctx, d_bases, h_read_start[nreads], pr));
  return align_checked(ctx, idx, p, pr, d_read_start, h_read_start, nreads, out);
}

int mr_align_batch_device_packed(mr_context* ctx, mr_index* idx, const mr_params* p, const uint64_t* d_codes, const uint64_t* d_nmask,
                                 const uint64_t* d_read_start, const uint64_t* h_read_start, uint32_t nreads, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!d_codes || !d_nmask) return ctx->fail(MR_EINVAL, "mr_align_batch: null argument");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  return align_checked(ctx, idx, p, make_packed(d_codes, d_nmask), d_read_start, h_read_start, nreads, out);
}

int mr_align_batch(mr_context* ctx, mr_index* idx, const mr_params* p, const char* bases, const uint64_t* read_start,
                   uint32_t nreads, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!bases || !read_start) return ctx->fail(MR_EINVAL, "mr_align_batch: null argument");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  const uint64_t T = read_start[nreads];
  MR_TRY(ws.bases.ensure(ctx, T + 64));
  MR_TRY(ws.read_start.ensure(ctx, ((size_t)nreads + 1) * 8));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.bases.p, bases, T, cudaMemcpyHostToDevice, ctx->stream));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.read_start.p, read_start, ((size_t)nreads + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  return mr_align_batch_device(ctx, idx, p, ws.bases.as<char>(), ws.read_start.as<uint64_t>(), read_start, nreads, out);
}

int mr_align_batch_packed(mr_context* ctx, mr_index* idx, const mr_params* p, const uint64_t* codes, const uint64_t* nmask,
                          const uint64_t* read_start, uint32_t nreads, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!codes || !nmask || !read_start) return ctx->fail(MR_EINVAL, "mr_align_batch: null argument");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  const uint64_t T = read_start[nreads];
  const uint64_t cwords = mr_packed_code_words(T), mwords = mr_packed_mask_words(T);
  MR_TRY(ws.codes.ensure(ctx, cwords * 8)); MR_TRY(ws.nmask.ensure(ctx, mwords * 8));
  MR_TRY(ws.read_start.ensure(ctx, ((size_t)nreads + 1) * 8));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.codes.p, codes, cwords * 8, cudaMemcpyHostToDevice, ctx->stream));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.nmask.p, nmask, mwords * 8, cudaMemcpyHostToDevice, ctx->stream));
  MR_CUDA(ctx, cudaMemcpyAsync(ws.read_start.p, read_start, ((size_t)nreads + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  return align_checked(ctx, idx, p, make_packed(ws.codes.as<uint64_t>(), ws.nmask.as<uint64_t>()), ws.read_start.as<uint64_t>(), read_start, nreads, out);
}

// Overlap graph of coords rows that come from the caller (host memory) instead of from the aligner:
// replaces overlap_graph::thread::reset + traverse (overlap_graph.hpp:177-198, overlap_graph.cc:7-59)
// as longest_path_overlap_graph2.cc:46-49 calls them on the rows of a coords file.
int mr_graph_batch(mr_context* ctx, const mr_params* p, const mr_result_view* rows, const uint32_t* read_len,
                   const uint32_t* path_ids, const uint64_t* path_off, uint32_t npaths,
                   const int32_t* unitig_len, uint32_t n_unitigs, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!p || !rows || !out || !read_len || !path_ids || !path_off || !unitig_len)
    return ctx->fail(MR_EINVAL, "mr_graph_batch: null argument");
  if(!p->unitigs_k || !n_unitigs) return ctx->fail(MR_EINVAL, "mr_graph_batch: the overlap graph needs unitig lengths and -k");
  *out = nullptr;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  ws.graph_stamp = ws.rows_stamp = 0;
  cudaStream_t st = ctx->stream;
  const uint32_t nreads = rows->nreads;
  const uint64_t S = rows->ncoords, Sc = std::max<uint64_t>(S, 1);
  if(S >= (1ULL << 31)) return ctx->fail(MR_ELIMIT, "mr_graph_batch: too many rows in one batch");
  if(rows->read_coords[0] != 0 || rows->read_coords[nreads] != S) return ctx->fail(MR_EINVAL, "mr_graph_batch: read_coords must span [0, ncoords]");
  uint64_t info_total = 0;
  for(uint64_t i = 0; i < path_off[npaths]; ++i)
    if((path_ids[i] >> 1) >= n_unitigs)
      return ctx->fail(MR_EINVAL, "mr_graph_batch: a path refers to a k-unitig that the unitig table does not have");
  for(uint64_t i = 0; i < S; ++i) {
    if(rows->sr[i] >= npaths) return ctx->fail(MR_EINVAL, "mr_graph_batch: row refers to a path that was not given");
    if(rows->info_len[i]) info_total = std::max<uint64_t>(info_total, rows->info_off[i] + rows->info_len[i]);
  }
  std::vector<uint32_t> row_read(Sc, 0);
  int max_rows = 0;
  for(uint32_t r = 0; r < nreads; ++r) {
    if(rows->read_coords[r + 1] < rows->read_coords[r] || rows->read_coords[r + 1] > S) return ctx->fail(MR_EINVAL, "mr_graph_batch: read_coords must be non-decreasing");
    max_rows = (int)std::max<uint64_t>(max_rows, std::min<uint64_t>(rows->read_coords[r + 1] - rows->read_coords[r], 0x7fffffff));
    for(uint64_t i = rows->read_coords[r]; i < rows->read_coords[r + 1]; ++i) row_read[i] = r;
  }
  ctx->timers.clear();
  phase_timer timer(ctx);
  timer.begin("rows upload");
  std::unique_ptr<mr_result> res(new mr_result);
  res->ctx = ctx;
  memset(&res->view, 0, sizeof(res->view));
  res->view.nreads = nreads;
  coords_soa fin;
  MR_TRY(setup_final_rows(ctx, ws, Sc, fin));
  MR_TRY(ws.read_coords.ensure(ctx, ((size_t)nreads + 2) * 8));
  MR_TRY(ws.read_len.ensure(ctx, ((size_t)nreads + 1) * 4));
  MR_TRY(ws.kinfo.ensure(ctx, (info_total + 1) * 4)); MR_TRY(ws.binfo.ensure(ctx, (info_total + 1) * 4));
  MR_TRY(ws.path_ids.ensure(ctx, (path_off[npaths] + 1) * 4)); MR_TRY(ws.path_off.ensure(ctx, ((size_t)npaths + 1) * 8));
  MR_TRY(ws.path_ulen.ensure(ctx, (size_t)n_unitigs * 4));
  auto push = [&](void* dst, const void* src, uint64_t bytes) { if(bytes) cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st); };
  push(ws.read_coords.p, rows->read_coords, ((uint64_t)nreads + 1) * 8);
  push(ws.read_len.p, read_len, (uint64_t)nreads * 4);
  push(fin.rs, rows->rs, S * 4); push(fin.re, rows->re, S * 4); push(fin.qs, rows->qs, S * 4); push(fin.qe, rows->qe, S * 4);
  push(fin.nb_mers, rows->nb_mers, S * 4);
  push(fin.pb_cons, rows->pb_cons, S * 4); push(fin.sr_cons, rows->sr_cons, S * 4);
  push(fin.pb_cover, rows->pb_cover, S * 4); push(fin.sr_cover, rows->sr_cover, S * 4);
  push(fin.ql, rows->ql, S * 4); push(fin.sr, rows->sr, S * 4); push(fin.read, row_read.data(), S * 4);
  push(fin.rn, rows->rn, S); push(fin.use_bwd, rows->use_bwd, S);
  push(fin.stretch, rows->stretch, S * 8); push(fin.offset, rows->offset, S * 8); push(fin.avg_err, rows->avg_err, S * 8);
  push(fin.info_off, rows->info_off, S * 8); push(fin.info_len, rows->info_len, S * 4);
  push(ws.kinfo.p, rows->kmers_info, info_total * 4); push(ws.binfo.p, rows->bases_info, info_total * 4);
  push(ws.path_ids.p, path_ids, path_off[npaths] * 4); push(ws.path_off.p, path_off, ((uint64_t)npaths + 1) * 8);
  push(ws.path_ulen.p, unitig_len, (uint64_t)n_unitigs * 4);
  MR_CUDA(ctx, cudaGetLastError());
  timer.next("overlap graph");
  graph_args GA;
  memset(&GA, 0, sizeof(GA));
  GA.nreads = nreads; GA.read_coords = ws.read_coords.as<uint64_t>(); GA.read_len = ws.read_len.as<uint32_t>(); GA.c = fin;
  GA.kinfo = ws.kinfo.as<int32_t>(); GA.binfo = ws.binfo.as<int32_t>();
  GA.unitig_ids = ws.path_ids.as<uint32_t>(); GA.unitig_off = ws.path_off.as<uint64_t>();
  GA.unitig_len = ws.path_ulen.as<int32_t>(); GA.n_unitigs = n_unitigs; GA.unitigs_k = p->unitigs_k;
  GA.overlap_play = p->overlap_play; GA.errors = p->errors; GA.bases = p->bases; GA.warp_max_rows = big_rows_threshold();
  MR_TRY(setup_graph_nodes(ctx, ws, Sc, GA));
  if(S) MR_TRY(launch_graph(ctx, ws, GA, S, max_rows));
  timer.next("result download");
  MR_TRY(download_rows(ctx, ws, res.get(), fin, nreads, S, info_total, &GA));
  timer.end();
  MR_CUDA(ctx, ctx->wait(st));
  timer.collect();
  remember_rows(ws, res.get(), fin, nreads, &GA, S, max_rows);
  *out = res.release();
  return MR_OK;
}

// Staged batches: the host -> device copy of batch i + 1 runs on its own stream while the kernels
// of batch i run.  mr_stage_batch may be called from another host thread than the one that aligns
// (a pageable source makes the copy call block; a pinned one, mr_host_pin, returns at once).
static int stage_impl(mr_context* ctx, const char* bases, const uint64_t* codes, const uint64_t* nmask, const uint64_t* read_start,
                      uint32_t nreads, mr_staged** out) {
  *out = nullptr;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  if(!ctx->ws) ctx->ws = new mr_workspace;
  mr_workspace& ws = *ctx->ws;
  std::unique_ptr<mr_staged> s;
  {
    std::lock_guard<std::mutex> lock(ws.pool_mutex);
    if(!ws.staged_pool.empty()) { s.reset(ws.staged_pool.back()); ws.staged_pool.pop_back(); }
  }
  if(!s) {
    s.reset(new mr_staged);
    s->ctx = ctx;
    MR_CUDA(ctx, cudaEventCreateWithFlags(&s->ready, cudaEventDisableTiming));
  }
  const uint64_t T = read_start[nreads];
  MR_TRY(s->read_start.ensure(ctx, ((size_t)nreads + 1) * 8));
  s->h_read_start.assign(read_start, read_start + nreads + 1);
  s->nreads = nreads;
  s->packed = bases == nullptr;
  if(bases) {
    MR_TRY(s->bases.ensure(ctx, T + 64));
    MR_CUDA(ctx, cudaMemcpyAsync(s->bases.p, bases, T, cudaMemcpyHostToDevice, ctx->copy_stream));
  } else {
    const uint64_t cwords = mr_packed_code_words(T), mwords = mr_packed_mask_words(T);
    MR_TRY(s->bases.ensure(ctx, (cwords + (cwords & 1) + mwords) * 8));          // mask words start 16-byte aligned
    MR_CUDA(ctx, cudaMemcpyAsync(s->bases.p, codes, cwords * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
    MR_CUDA(ctx, cudaMemcpyAsync(s->bases.as<uint64_t>() + cwords + (cwords & 1), nmask, mwords * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
  }
  MR_CUDA(ctx, cudaMemcpyAsync(s->read_start.p, s->h_read_start.data(), ((size_t)nreads + 1) * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
  MR_CUDA(ctx, cudaEventRecord(s->ready, ctx->copy_stream));
  *out = s.release();
  return MR_OK;
}

int mr_stage_batch(mr_context* ctx, const char* bases, const uint64_t* read_start, uint32_t nreads, mr_staged** out) {
  if(!ctx) return MR_EINVAL;
  if(!bases || !read_start || !out) return ctx->fail(MR_EINVAL, "mr_stage_batch: null argument");
  return stage_impl(ctx, bases, nullptr, nullptr, read_start, nreads, out);
}

int mr_stage_batch_packed(mr_context* ctx, const uint64_t* codes, const uint64_t* nmask, const uint64_t* read_start, uint32_t nreads,
                          mr_staged** out) {
  if(!ctx) return MR_EINVAL;
  if(!codes || !nmask || !read_start || !out) return ctx->fail(MR_EINVAL, "mr_stage_batch: null argument");
  return stage_impl(ctx, nullptr, codes, nmask, read_start, nreads, out);
}

void mr_staged_free(mr_staged* s) {
  if(!s) return;
  cudaSetDevice(s->ctx->device);
  cudaEventSynchronize(s->ready);
  mr_workspace* ws = s->ctx->ws;
  if(ws) {
    std::lock_guard<std::mutex> lock(ws->pool_mutex);
    if(ws->staged_pool.size() < 4) { ws->staged_pool.push_back(s); return; }
  }
  delete s;
}

int mr_align_staged(mr_context* ctx, mr_index* idx, const mr_params* p, mr_staged* s, mr_result** out) {
  if(!ctx) return MR_EINVAL;
  if(!s || s->ctx != ctx) return ctx->fail(MR_EINVAL, "mr_align_staged: the batch was staged on another context");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  MR_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, s->ready, 0));
  int rc;
  if(s->packed) {
    const uint64_t cwords = mr_packed_code_words(s->h_read_start[s->nreads]);
    rc = mr_align_batch_device_packed(ctx, idx, p, s->bases.as<uint64_t>(), s->bases.as<uint64_t>() + cwords + (cwords & 1),
                                      s->read_start.as<uint64_t>(), s->h_read_start.data(), s->nreads, out);
  } else rc = mr_align_batch_device(ctx, idx, p, s->bases.as<char>(), s->read_start.as<uint64_t>(), s->h_read_start.data(), s->nreads, out);
  mr_staged_free(s);
  return rc;
}

void mr_result_free(mr_result* r) {
  if(!r) return;
  cudaSetDevice(r->ctx->device);
  if(r->host) {
    bool kept = false;
    if(r->ctx->ws) {
      std::lock_guard<std::mutex> lock(r->ctx->ws->pool_mutex);
      if(r->ctx->ws->pinned_pool.size() < 4) { r->ctx->ws->pinned_pool.push_back(r->host); kept = true; }
    }
    if(!kept) delete r->host;
  }
  delete r;
}

int mr_result_get(const mr_result* r, mr_result_view* view) {
  if(!r || !view) return MR_EINVAL;
  *view = r->view;
  return MR_OK;
}

int mr_result_taps(const mr_result* r, uint64_t* ngroups, const int64_t** groups, uint64_t* noffsets, const int32_t** offsets,
                   uint64_t* nlis, const uint32_t** lis) {
  if(!r) return MR_EINVAL;
  if(ngroups) *ngroups = r->tap_groups.size() / 6;
  if(groups) *groups = r->tap_groups.data();
  if(noffsets) *noffsets = r->tap_offsets.size() / 2;
  if(offsets) *offsets = r->tap_offsets.data();
  if(nlis) *nlis = r->tap_lis.size();
  if(lis) *lis = r->tap_lis.data();
  return MR_OK;
}

} // extern "C"

// Device-wide building blocks written for this library: exclusive scan and a stable LSD radix
// sort (key/value).  Both are plain HBM-streaming kernels: every pass reads its input once in
// fully coalesced 16 KiB tiles and writes once; the roofline for them is the copy bandwidth.
#pragma once
#include "common.cuh"
#include <algorithm>

namespace prim {

constexpr int kScanThreads = 256;
constexpr int kScanItems   = 16;
constexpr int kScanTile    = kScanThreads * kScanItems;   // 4096 elements per CTA

// ---- block helpers -----------------------------------------------------------------------------
// exclusive scan of one uint64 per thread across a 256-thread CTA; returns the CTA total in `total`
__device__ __forceinline__ uint64_t block_exclusive_scan_256(uint64_t v, uint64_t* smem_warp /*[8]*/, uint64_t& total) {
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t inc = v;
#pragma unroll
  for(int d = 1; d < 32; d <<= 1) {
    const uint64_t o = __shfl_up_sync(MR_FULL_MASK, inc, d);
    if(lane >= (unsigned)d) inc += o;
  }
  if(lane == 31) smem_warp[warp] = inc;
  __syncthreads();
  uint64_t wprefix = 0, tot = 0;
#pragma unroll
  for(int w = 0; w < 8; ++w) {
    const uint64_t s = smem_warp[w];
    if((unsigned)w < warp) wprefix += s;
    tot += s;
  }
  total = tot;
  __syncthreads();
  return wprefix + inc - v;
}

// ---- CTA bitonic sort of an index array in shared memory ---------------------------------------------
// idx[0 .. m), m a power of two; less(a, b) is a strict total order on the entries (callers break ties by the
// entry itself, so the result does not depend on the network); entries equal to kPad sort last.  All
// threads of the CTA must call it.  m log2(m)^2 / 4 compare-exchanges: 0.3 M for 4096 entries, where ranking
// by counting costs 16 M comparisons.
constexpr uint32_t kPad = 0xffffffffu;
template<typename Less>
__device__ __forceinline__ void bitonic_sort_idx(uint32_t* idx, int m, Less less) {
  for(int k = 2; k <= m; k <<= 1) {
    for(int j = k >> 1; j > 0; j >>= 1) {
      for(int t = (int)threadIdx.x; t < (m >> 1); t += (int)blockDim.x) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));      // bit j clear
        const int l = i | j;
        const uint32_t a = idx[i], b = idx[l];
        const bool b_first = b != kPad && (a == kPad || less(b, a));
        const bool a_first = a != kPad && (b == kPad || less(a, b));
        if((i & k) == 0 ? b_first : a_first) { idx[i] = b; idx[l] = a; }
      }
      __syncthreads();
    }
  }
}

// ---- exclusive scan: out[i] = sum_{j<i} in(j), in() yields uint32/uint64 ------------------------
template<typename In>
__global__ void __launch_bounds__(kScanThreads) scan_reduce_kernel(In in, uint64_t n, uint64_t* __restrict__ block_sums) {
  __shared__ uint64_t sw[8];
  const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
  uint64_t s = 0;
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) {          // striped: coalesced reads
    const uint64_t idx = base + (uint64_t)i * kScanThreads + threadIdx.x;
    if(idx < n) s += in(idx);
  }
  uint64_t total;
  (void)block_exclusive_scan_256(s, sw, total);
  if(threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single CTA: exclusive scan of the per-tile sums in place, grand total to *total
static __global__ void __launch_bounds__(1024) scan_blocksums_kernel(uint64_t* __restrict__ block_sums, uint32_t nblocks, uint64_t* __restrict__ total) {
  __shared__ uint64_t sw[32];
  __shared__ uint64_t carry_s;
  if(threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for(uint32_t base = 0; base < nblocks; base += 1024) {
    const uint32_t idx = base + threadIdx.x;
    const uint64_t v = idx < nblocks ? block_sums[idx] : 0;
    uint64_t inc = v;
#pragma unroll
    for(int d = 1; d < 32; d <<= 1) {
      const uint64_t o = __shfl_up_sync(MR_FULL_MASK, inc, d);
      if(lane >= (unsigned)d) inc += o;
    }
    if(lane == 31) sw[warp] = inc;
    __syncthreads();
    uint64_t wprefix = 0, tot = 0;
    for(int w = 0; w < 32; ++w) { const uint64_t s = sw[w]; if((unsigned)w < warp) wprefix += s; tot += s; }
    const uint64_t carry = carry_s;
    if(idx < nblocks) block_sums[idx] = carry + wprefix + inc - v;
    __syncthreads();
    if(threadIdx.x == 0) carry_s = carry + tot;
    __syncthreads();
  }
  if(threadIdx.x == 0 && total) *total = carry_s;
}

template<typename In, typename OutT>
__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(In in, uint64_t n, const uint64_t* __restrict__ block_sums, OutT* __restrict__ out) {
  __shared__ uint64_t sw[8];
  __shared__ uint64_t stage[kScanTile];          // transposes striped loads into blocked order (32 KiB)
  const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) {
    const uint32_t t = i * kScanThreads + threadIdx.x;
    const uint64_t idx = base + t;
    stage[t] = idx < n ? (uint64_t)in(idx) : 0;
  }
  __syncthreads();
  uint64_t v[kScanItems], s = 0;
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) { v[i] = stage[threadIdx.x * kScanItems + i]; s += v[i]; }
  uint64_t total;
  uint64_t run = block_exclusive_scan_256(s, sw, total) + block_sums[blockIdx.x];
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) { stage[threadIdx.x * kScanItems + i] = run; run += v[i]; }
  __syncthreads();
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) {
    const uint32_t t = i * kScanThreads + threadIdx.x;
    const uint64_t idx = base + t;
    if(idx < n) out[idx] = (OutT)stage[t];
  }
}

// positions of the set flags: out[k] = index of the k-th i with in(i) != 0 (in() yields 0 / 1).
// Same tile walk as scan_apply_kernel, but only the flagged positions are written.
template<typename In>
__global__ void __launch_bounds__(kScanThreads) flag_positions_kernel(In in, uint64_t n, const uint64_t* __restrict__ block_sums,
                                                                       uint64_t* __restrict__ out) {
  __shared__ uint64_t sw[8];
  __shared__ uint8_t stage[kScanTile];
  const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) {
    const uint32_t t = i * kScanThreads + threadIdx.x;
    const uint64_t idx = base + t;
    stage[t] = idx < n ? (uint8_t)in(idx) : 0;
  }
  __syncthreads();
  uint32_t flags = 0, s = 0;
#pragma unroll
  for(int i = 0; i < kScanItems; ++i) { const uint32_t f = stage[threadIdx.x * kScanItems + i]; flags |= f << i; s += f; }
  uint64_t total;
  uint64_t run = block_exclusive_scan_256(s, sw, total) + block_sums[blockIdx.x];
#pragma unroll
  for(int i = 0; i < kScanItems; ++i)
    if((flags >> i) & 1) out[run++] = base + (uint64_t)threadIdx.x * kScanItems + i;
}

// out[] as above; *d_total (device) and block_sums scratch as in exclusive_scan.  Two launches +
// the single-CTA scan of the tile sums; the caller reads *d_total before sizing `out`, so the
// positions are written by a separate call.
template<typename In>
int flag_count(mr_context* ctx, In in, uint64_t n, dev_buf& scratch, uint64_t* d_total) {
  const uint32_t nblocks = div_up(n, kScanTile);
  if(n == 0) { MR_CUDA(ctx, cudaMemsetAsync(d_total, 0, sizeof(uint64_t), ctx->stream)); return MR_OK; }
  MR_TRY(scratch.ensure(ctx, ((size_t)nblocks + 1) * sizeof(uint64_t)));
  scan_reduce_kernel<In><<<nblocks, kScanThreads, 0, ctx->stream>>>(in, n, scratch.as<uint64_t>());
  MR_LAUNCHED(ctx);
  scan_blocksums_kernel<<<1, 1024, 0, ctx->stream>>>(scratch.as<uint64_t>(), nblocks, d_total);
  MR_LAUNCHED(ctx);
  return MR_OK;
}
template<typename In>
int flag_positions(mr_context* ctx, In in, uint64_t n, dev_buf& scratch, uint64_t* out) {
  if(n == 0) return MR_OK;
  flag_positions_kernel<In><<<div_up(n, kScanTile), kScanThreads, 0, ctx->stream>>>(in, n, scratch.as<uint64_t>(), out);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

struct ptr_in_u32 { const uint32_t* p; __device__ uint64_t operator()(uint64_t i) const { return p[i]; } };
struct ptr_in_u64 { const uint64_t* p; __device__ uint64_t operator()(uint64_t i) const { return p[i]; } };

// scratch: block_sums buffer (>= div_up(n, 4096) + 1 uint64).  total (device pointer) may be null.
template<typename In, typename OutT>
int exclusive_scan(mr_context* ctx, In in, uint64_t n, OutT* out, dev_buf& scratch, uint64_t* d_total) {
  const uint32_t nblocks = div_up(n, kScanTile);
  if(n == 0) {
    if(d_total) MR_CUDA(ctx, cudaMemsetAsync(d_total, 0, sizeof(uint64_t), ctx->stream));
    return MR_OK;
  }
  MR_TRY(scratch.ensure(ctx, ((size_t)nblocks + 1) * sizeof(uint64_t)));
  uint64_t* bs = scratch.as<uint64_t>();
  scan_reduce_kernel<In><<<nblocks, kScanThreads, 0, ctx->stream>>>(in, n, bs);
  MR_LAUNCHED(ctx);
  scan_blocksums_kernel<<<1, 1024, 0, ctx->stream>>>(bs, nblocks, d_total);
  MR_LAUNCHED(ctx);
  scan_apply_kernel<In, OutT><<<nblocks, kScanThreads, 0, ctx->stream>>>(in, n, bs, out);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

// ---- stable LSD radix sort ----------------------------------------------------------------------
constexpr int kSortBits    = 8;
constexpr int kSortRadix   = 1 << kSortBits;
constexpr int kSortThreads = 256;
constexpr int kSortWarps   = kSortThreads / 32;
constexpr int kSortItems   = 16;
constexpr int kSortTile    = kSortThreads * kSortItems;   // 4096 keys per CTA

// kBits: width of the digit of this pass (at most kSortBits); a key range that is not a multiple of 8 bits is
// cut into equal digits (14 bits: 7 + 7, 21 bits: 7 + 7 + 7) -- half as many buckets per pass means runs
// twice as long in the scattered stores
template<typename K, int kBits>
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const K* __restrict__ keys, uint64_t n, int shift,
                                                                   uint32_t* __restrict__ table, uint32_t nblocks) {
  constexpr int kRadix = 1 << kBits;
  __shared__ uint32_t h[kRadix];
  if(threadIdx.x < kRadix) h[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t base = (uint64_t)blockIdx.x * kSortTile;
#pragma unroll
  for(int i = 0; i < kSortItems; ++i) {
    const uint64_t idx = base + (uint64_t)i * kSortThreads + threadIdx.x;
    if(idx < n) atomicAdd(&h[(unsigned)(keys[idx] >> shift) & (kRadix - 1)], 1u);
  }
  __syncthreads();
  if(threadIdx.x < kRadix) table[(uint64_t)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];   // digit-major
}

// Each warp owns a contiguous 256-key slice of the tile and walks it 32 keys at a time, so the
// rank of a key among equal digits is (earlier warps) + (earlier rounds of this warp) + (lower
// lanes of this round): order preserving, hence stable.
// kScatterThreads threads rank a tile of kSortTile keys, 8 each.  256 threads x 16 keys keeps 16 keys and ranks per
// thread in registers and leaves the SM at ~22 % occupancy with every warp waiting on its loads (ncu:
// long_scoreboard); 512 x 8 halves the registers and doubles the warps in flight.
constexpr int kScatterThreads = 512;
template<typename K, typename V, int kBits>
__global__ void __launch_bounds__(kScatterThreads) radix_scatter_kernel(const K* __restrict__ kin, const V* __restrict__ vin,
                                                                  K* __restrict__ kout, V* __restrict__ vout,
                                                                  uint64_t n, int shift,
                                                                  const uint64_t* __restrict__ offsets, uint32_t nblocks) {
  constexpr int kRadix = 1 << kBits, kWarps = kScatterThreads / 32, kItems = kSortTile / kScatterThreads;
  __shared__ uint32_t cnt[kWarps][kRadix];
  __shared__ uint32_t wrel[kWarps][kRadix];       // first slot of warp w's keys with digit d, relative to dbase[d]
  __shared__ uint64_t dbase[kRadix];              // first slot of this tile's keys with digit d
  for(int i = threadIdx.x; i < kWarps * kRadix; i += kScatterThreads) (&cnt[0][0])[i] = 0;
  __syncthreads();
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t base = (uint64_t)blockIdx.x * kSortTile + (uint64_t)warp * (32 * kItems);
  const unsigned lt = lanemask_lt();
  K        key[kItems];
  uint32_t rank[kItems];
#pragma unroll
  for(int i = 0; i < kItems; ++i) {
    const uint64_t idx = base + (uint64_t)i * 32 + lane;
    const bool valid = idx < n;
    key[i] = valid ? kin[idx] : (K)0;
    const unsigned d = valid ? ((unsigned)(key[i] >> shift) & (kRadix - 1)) : (unsigned)kRadix;
    const unsigned peers  = __match_any_sync(MR_FULL_MASK, d);
    const unsigned leader = __ffs(peers) - 1;
    unsigned b = 0;
    if(valid && lane == leader) { b = cnt[warp][d]; cnt[warp][d] = b + __popc(peers); }
    b = __shfl_sync(MR_FULL_MASK, b, leader);
    rank[i] = b + __popc(peers & lt);
    __syncwarp();
  }
  __syncthreads();
  for(unsigned d = threadIdx.x; d < (unsigned)kRadix; d += kScatterThreads) {
    dbase[d] = offsets[(uint64_t)d * nblocks + blockIdx.x];
    uint32_t run = 0;
#pragma unroll
    for(int w = 0; w < kWarps; ++w) { wrel[w][d] = run; run += cnt[w][d]; }
  }
  __syncthreads();
#pragma unroll
  for(int i = 0; i < kItems; ++i) {
    const uint64_t idx = base + (uint64_t)i * 32 + lane;
    if(idx < n) {
      const unsigned d = (unsigned)(key[i] >> shift) & (kRadix - 1);
      const uint64_t dst = dbase[d] + wrel[warp][d] + rank[i];
      kout[dst] = key[i];
      vout[dst] = vin[idx];
    }
  }
}

struct sort_scratch {
  dev_buf table;     // uint32[radix * nblocks]
  dev_buf offsets;   // uint64[radix * nblocks]
  dev_buf scan;      // scan scratch
};

// one pass on the digit [shift, shift + kBits)
template<typename K, typename V, int kBits>
int radix_pass(mr_context* ctx, const K* kin, const V* vin, K* kout, V* vout, uint64_t n, int shift, sort_scratch& s) {
  const uint32_t nblocks = div_up(n, kSortTile);
  const uint64_t tsize = ((uint64_t)1 << kBits) * nblocks;
  radix_hist_kernel<K, kBits><<<nblocks, kSortThreads, 0, ctx->stream>>>(kin, n, shift, s.table.as<uint32_t>(), nblocks);
  MR_LAUNCHED(ctx);
  MR_TRY((exclusive_scan<ptr_in_u32, uint64_t>(ctx, ptr_in_u32{ s.table.as<uint32_t>() }, tsize, s.offsets.as<uint64_t>(), s.scan, nullptr)));
  radix_scatter_kernel<K, V, kBits><<<nblocks, kScatterThreads, 0, ctx->stream>>>(kin, vin, kout, vout, n, shift, s.offsets.as<uint64_t>(), nblocks);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

// Sorts (k0,v0) by key bits [lo_bit, hi_bit) ascending, stable.  k1/v1 are same-sized alternates.
// On return *result_in_first tells whether the sorted data sits in (k0,v0) or (k1,v1).
template<typename K, typename V>
int radix_sort_pairs(mr_context* ctx, K* k0, V* v0, K* k1, V* v1, uint64_t n, int lo_bit, int hi_bit,
                     sort_scratch& s, bool* result_in_first) {
  bool first = true;
  if(n == 0 || hi_bit <= lo_bit) { *result_in_first = true; return MR_OK; }
  const uint32_t nblocks = div_up(n, kSortTile);
  const uint64_t tsize = (uint64_t)kSortRadix * nblocks;
  MR_TRY(s.table.ensure(ctx, tsize * sizeof(uint32_t)));
  MR_TRY(s.offsets.ensure(ctx, tsize * sizeof(uint64_t)));
  const int bits = hi_bit - lo_bit, passes = (bits + kSortBits - 1) / kSortBits;
  int shift = lo_bit;
  for(int p = 0; p < passes; ++p) {
    // digits of kSortBits bits, the last one narrower: faster than equal digits (DESIGN.md §4)
    int w = std::min(kSortBits, hi_bit - shift);
    K* kin = first ? k0 : k1; V* vin = first ? v0 : v1;
    K* kout = first ? k1 : k0; V* vout = first ? v1 : v0;
    switch(w) {
    case 8: MR_TRY((radix_pass<K, V, 8>(ctx, kin, vin, kout, vout, n, shift, s))); break;
    case 7: MR_TRY((radix_pass<K, V, 7>(ctx, kin, vin, kout, vout, n, shift, s))); break;
    case 6: MR_TRY((radix_pass<K, V, 6>(ctx, kin, vin, kout, vout, n, shift, s))); break;
    case 5: MR_TRY((radix_pass<K, V, 5>(ctx, kin, vin, kout, vout, n, shift, s))); break;
    default: MR_TRY((radix_pass<K, V, 4>(ctx, kin, vin, kout, vout, n, shift, s))); w = std::min(w, 4); break;
    }
    shift += w;
    first = !first;
  }
  // digits narrower than 4 bits are rounded up to 4: the extra key bits above hi_bit are sorted too, which is
  // harmless for every caller (they are part of the same key and equal within what the caller groups by)
  *result_in_first = first;
  return MR_OK;
}

} // namespace prim

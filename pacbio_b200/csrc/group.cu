// Grouping of a batch's hits by (read, super-read): frags_pos_type of coarse_aligner.hpp:14 /
// coarse_aligner.cc:132-138, where the reference appends every hit to an unordered_map of per-super-read
// vectors while it walks one read.
//
// The expansion emits the hits read-major, in the order the reference visits them (read position, forward
// list before reverse list, suffix-array order), so the hits of one read are one contiguous slice of the hit
// arrays and grouping is a STABLE sort of that slice on the super-read index alone.  One CTA per read.
//
// (1) A read of the usual kind has a few thousand hits: the whole slice fits the shared memory of one SM.  The CTA
//   * pulls the slice's payloads into shared memory with one bulk asynchronous copy (TMA engine, completes on
//     an mbarrier while the CTA is busy with the keys),
//   * turns every key into (super-read << idx_bits | position in the slice), a 32-bit word,
//   * sorts those words with an LSD radix sort that never leaves shared memory (7-bit digits; every warp ranks
//     a contiguous piece 32 keys at a time with match_any, so the order among equal digits is the input order),
//   * writes keys and payloads back in sorted order, fully coalesced, together with one byte per hit that
//     says whether a new (read, super-read) group starts there.
//   Per hit that is 16 bytes read and 17 written, against (8 + 32) bytes per pass of a device-wide radix sort
//   plus 16 for the group heads: 33 instead of 96 bytes on the yeast-size index (14-bit super-read index).
//
// (2) A read whose hits do not fit (reads inside repeats; every read of the human-size shape, 10^5 hits each) is
//   first cut by the top 7 bits of the super-read index: one stable counting pass of the CTA over the slice, out
//   of global memory, 2048 or 4096 hits at a time with the running bucket offsets in shared memory.  Consecutive
//   buckets are then sorted as in (1), as many at a time as fit, on the remaining low bits (relative to the first
//   bucket's base, so the words stay 32 bit).  73 bytes per hit instead of the 136 of three device-wide passes
//   over a 21-bit index.
//
// (3) What is left -- a bucket that still does not fit, an index of more than 2^25 super-reads -- is sorted by
//   LSD passes of the same counting routine, ping-pong between the two buffer pairs.
//
// Hits whose k-mer straddles two super-reads carry the super-read index nseq_all: they sort to the end of
// their read's slice and form a group of their own, which the chaining kernels skip (chain.cu,
// classify_groups_kernel).
#include "align.cuh"
#include "group.cuh"

namespace {

constexpr int kGsRounds  = 16;              // keys per thread of the in-shared-memory sort
constexpr int kGsDigit   = 7;
constexpr int kGsRadix   = 1 << kGsDigit;
constexpr int kFbRounds  = 4;               // keys per thread and chunk of the passes out of global memory

template<int kThreads>
struct gs_layout {
  static constexpr int kWarps = kThreads / 32;
  static constexpr int kCap   = kThreads * kGsRounds;
  static constexpr size_t pay_off = 0;                                             // uint64[kCap + 2], 16-byte aligned
  static constexpr size_t arr_off = pay_off + (size_t)(kCap + 2) * 8;              // uint32[kCap]
  static constexpr size_t cnt_off = arr_off + (size_t)kCap * 4;                    // uint32[kWarps][kGsRadix]
  static constexpr size_t tot_off = cnt_off + (size_t)kWarps * kGsRadix * 4;       // uint32[kGsRadix]
  static constexpr size_t dbs_off = tot_off + kGsRadix * 4;                        // uint32[kGsRadix]
  static constexpr size_t bsz_off = dbs_off + kGsRadix * 4;                        // uint32[kGsRadix]: bucket sizes of (2)
  static constexpr size_t bst_off = bsz_off + kGsRadix * 4;                        // uint32[kGsRadix]: bucket starts of (2)
  static constexpr size_t wsm_off = bst_off + kGsRadix * 4;                        // uint32[4]
  static constexpr size_t cbs_off = wsm_off + 16;                                  // uint32[kGsRadix]: a chunk's bucket offsets
  static constexpr size_t bar_off = cbs_off + kGsRadix * 4;                        // uint64[4]: payload copy + three chunk buffers
  static constexpr size_t bytes   = bar_off + 32;
  // the passes out of global memory stage chunks of kFbRounds keys per thread in three buffers laid over spay and arr
  static_assert((size_t)3 * kThreads * kFbRounds * 16 <= cnt_off, "three chunk buffers of keys and payloads");
};

// the CTA's dynamic shared memory, addressed by constant offsets (no pointer registers: the kernel runs at 64 registers)
extern __shared__ __align__(16) unsigned char gs_raw[];
template<int kThreads>
struct gs_sm {
  typedef gs_layout<kThreads> L;
  static __device__ __forceinline__ uint64_t* spay()   { return reinterpret_cast<uint64_t*>(gs_raw + L::pay_off); }
  static __device__ __forceinline__ uint32_t* arr()    { return reinterpret_cast<uint32_t*>(gs_raw + L::arr_off); }
  static __device__ __forceinline__ uint32_t (*cnt())[kGsRadix] { return reinterpret_cast<uint32_t (*)[kGsRadix]>(gs_raw + L::cnt_off); }
  static __device__ __forceinline__ uint32_t* tot()    { return reinterpret_cast<uint32_t*>(gs_raw + L::tot_off); }
  static __device__ __forceinline__ uint32_t* dbase()  { return reinterpret_cast<uint32_t*>(gs_raw + L::dbs_off); }
  static __device__ __forceinline__ uint32_t* bsize()  { return reinterpret_cast<uint32_t*>(gs_raw + L::bsz_off); }
  static __device__ __forceinline__ uint32_t* bstart() { return reinterpret_cast<uint32_t*>(gs_raw + L::bst_off); }
  static __device__ __forceinline__ uint32_t* wsum()   { return reinterpret_cast<uint32_t*>(gs_raw + L::wsm_off); }
  static __device__ __forceinline__ uint32_t* cbase()  { return reinterpret_cast<uint32_t*>(gs_raw + L::cbs_off); }
  static __device__ __forceinline__ uint64_t* bar()    { return reinterpret_cast<uint64_t*>(gs_raw + L::bar_off); }       // payload copies of sort_range_smem
  static __device__ __forceinline__ uint64_t* cbar()   { return reinterpret_cast<uint64_t*>(gs_raw + L::bar_off) + 1; }   // [3]: chunk buffers of radix_pass_global
};

// rank of this lane's key among the keys of its warp's piece that have the same digit and come before it
// (earlier rounds through cnt, lower lanes of this round through the match mask); d == kGsRadix: no key
__device__ __forceinline__ uint32_t rank_round(uint32_t d, uint32_t* cnt_w, unsigned lt) {
  const unsigned peers = __match_any_sync(MR_FULL_MASK, d);
  const unsigned before = __popc(peers & lt);
  uint32_t b = 0;
  if(d < (uint32_t)kGsRadix) b = cnt_w[d];
  __syncwarp();
  if(before == 0 && d < (uint32_t)kGsRadix) cnt_w[d] = b + __popc(peers);
  __syncwarp();
  return b + before;
}

// the same on 16-bit counters (chunks of at most 4096 keys)
__device__ __forceinline__ uint32_t rank_round16(uint32_t d, uint16_t* cnt_w, unsigned lt) {
  const unsigned peers = __match_any_sync(MR_FULL_MASK, d);
  const unsigned before = __popc(peers & lt);
  uint32_t b = 0;
  if(d < (uint32_t)kGsRadix) b = cnt_w[d];
  __syncwarp();
  if(before == 0 && d < (uint32_t)kGsRadix) cnt_w[d] = (uint16_t)(b + __popc(peers));
  __syncwarp();
  return b + before;
}

// cnt[w][d] -> number of keys with digit d in the pieces of the warps before w; tot[d] = all of them; with
// kScan also dbase[d] = number of keys with a smaller digit.  Ends with a barrier.
template<int kWarps, bool kScan>
__device__ __forceinline__ void digit_prefix(uint32_t (*cnt)[kGsRadix], uint32_t* tot, uint32_t* dbase, uint32_t* wsum) {
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t run = 0, inc = 0;
  if(threadIdx.x < kGsRadix) {
#pragma unroll 8
    for(int w = 0; w < kWarps; ++w) { const uint32_t t = cnt[w][threadIdx.x]; cnt[w][threadIdx.x] = run; run += t; }
    tot[threadIdx.x] = run;
    if(kScan) {
      inc = run;
#pragma unroll
      for(int s = 1; s < 32; s <<= 1) { const uint32_t o = __shfl_up_sync(MR_FULL_MASK, inc, s); if(lane >= (unsigned)s) inc += o; }
      if(lane == 31) wsum[warp] = inc;
    }
  }
  __syncthreads();
  if(kScan) {
    if(threadIdx.x < kGsRadix) {
      uint32_t before = 0;
      for(unsigned w = 0; w < warp; ++w) before += wsum[w];
      dbase[threadIdx.x] = before + inc - run;
    }
    __syncthreads();
  }
}

// ---- (1): n <= capacity hits from (kin, pin) to (ko, po, head), sorted on (super-read - key_base), a number of
// key_bits bits.  kin == ko is allowed (everything is read before anything is written).  `phase` counts the uses
// of the CTA's mbarrier.  All threads call it; it starts and ends with the CTA in step.
template<int kThreads>
__device__ void sort_range_smem(const uint64_t* kin, const uint64_t* pin, uint64_t* ko, uint64_t* po, uint8_t* head,
                                uint32_t n, uint32_t key_base, int key_bits, uint32_t ib, uint64_t rhi, uint32_t& phase) {
  typedef gs_sm<kThreads> Sm;
  constexpr int kWarps = kThreads / 32;
  const unsigned warp = threadIdx.x >> 5, lt = lanemask_lt();
  uint32_t* arr = Sm::arr();
  // payloads: one bulk copy of the slice, widened to 16-byte bounds (the hit arrays are padded by two entries)
  const uint32_t skew = (uint32_t)(((uintptr_t)pin >> 3) & 1u);
  if(threadIdx.x == 0) {
    const uint32_t bytes = ((n + skew + 1) & ~1u) * 8u;
    mbar_expect_tx(Sm::bar(), bytes);
    bulk_copy_g2s(Sm::spay(), pin - skew, bytes, Sm::bar());
  }
#pragma unroll 4
  for(uint32_t j = threadIdx.x; j < n; j += kThreads) arr[j] = (((uint32_t)kin[j] - key_base) << ib) | j;
  __syncthreads();
  const uint32_t R = (n + kThreads - 1) / kThreads;           // rounds; warp w ranks positions [32 R w, 32 R (w + 1))
  const uint32_t piece = warp * 32 * R + (threadIdx.x & 31);
  const int passes = (key_bits + kGsDigit - 1) / kGsDigit;
  for(int p = 0; p < passes; ++p) {
    const int shift = (int)ib + p * kGsDigit;
    for(int i = threadIdx.x; i < kWarps * kGsRadix; i += kThreads) (&Sm::cnt()[0][0])[i] = 0;
    __syncthreads();
    uint32_t e[kGsRounds], rk[kGsRounds / 2];                 // ranks are below 2^14: two to a register
#pragma unroll
    for(int i = 0; i < kGsRounds; ++i) {
      if((i & 1) == 0) rk[i >> 1] = 0;
      if((uint32_t)i < R) {
        const uint32_t pos = piece + i * 32;
        const bool valid = pos < n;
        e[i] = valid ? arr[pos] : 0u;
        rk[i >> 1] |= rank_round(valid ? (e[i] >> shift) & (kGsRadix - 1) : (uint32_t)kGsRadix, Sm::cnt()[warp], lt) << (16 * (i & 1));
      }
    }
    __syncthreads();
    digit_prefix<kWarps, true>(Sm::cnt(), Sm::tot(), Sm::dbase(), Sm::wsum());
#pragma unroll
    for(int i = 0; i < kGsRounds; ++i) {
      if((uint32_t)i < R && piece + i * 32 < n) {
        const uint32_t d = (e[i] >> shift) & (kGsRadix - 1);
        arr[Sm::dbase()[d] + Sm::cnt()[warp][d] + ((rk[i >> 1] >> (16 * (i & 1))) & 0xffffu)] = e[i];
      }
    }
    __syncthreads();
  }
  mbar_wait(Sm::bar(), phase & 1u);
  ++phase;
  const uint32_t imask = (1u << ib) - 1;
#pragma unroll 4
  for(uint32_t j = threadIdx.x; j < n; j += kThreads) {
    const uint32_t x = arr[j], rel = x >> ib;
    ko[j] = rhi | (uint64_t)(key_base + rel);
    po[j] = Sm::spay()[skew + (x & imask)];
    head[j] = j == 0 || (arr[j - 1] >> ib) != rel;
  }
  __syncthreads();                                            // arr and spay may be overwritten by the next range
}

// ---- one stable counting pass of the CTA over (sk, sp)[0, n) -> (dk, dp)[0, n) on digit (key >> shift) & dmask,
// out of global memory.  With `keep` the digit histogram and its exclusive scan stay in bsize / bstart.
// After a histogram sweep over the keys, the slice is walked in chunks of kFbRounds keys per thread; the TMA engine
// copies chunk c + 2 (keys and payloads: two contiguous pieces) into one of three shared-memory buffers while the
// CTA ranks and scatters chunk c, two barriers per chunk.  `gc` numbers the chunks the CTA has staged so far: chunk
// g uses buffer g % 3, whose mbarrier is then in phase (g / 3) & 1.  Chunks are cut at even hit indices so that every
// bulk copy is 16-byte aligned (a slice that starts at an odd index gets one dead position in front).
template<int kThreads>
__device__ void radix_pass_global(const uint64_t* sk, const uint64_t* sp, uint64_t* dk, uint64_t* dp, uint32_t n,
                                  int shift, uint32_t dmask, bool keep, uint32_t& gc) {
  typedef gs_sm<kThreads> Sm;
  constexpr int kWarps = kThreads / 32, kChunk = kThreads * kFbRounds;
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, lt = lanemask_lt();
  uint32_t *tot = Sm::tot(), *gbase = Sm::dbase(), *cbase = Sm::cbase();
  uint16_t (*C)[kWarps][kGsRadix] = reinterpret_cast<uint16_t (*)[kWarps][kGsRadix]>(Sm::cnt());     // two sets of 16-bit counters
  for(int i = threadIdx.x; i < kGsRadix; i += kThreads) tot[i] = 0;
  for(int i = threadIdx.x; i < kWarps * kGsRadix; i += kThreads) (&C[0][0][0])[i] = 0;
  asm volatile("fence.proxy.async;" ::: "memory");       // what this CTA stored (global: the previous pass; shared: the buffers) before the bulk copies
  __syncthreads();
  const uint32_t skew = (uint32_t)(((uintptr_t)sk >> 3) & 1u);            // (sp has the same parity: same index, 256-byte aligned arrays)
  const uint64_t *ska = sk - skew, *spa = sp - skew;
  const uint64_t m = (uint64_t)n + skew;                                   // positions [skew, m) of the aligned slice are hits
  const uint32_t nchunks = (uint32_t)((m + kChunk - 1) / kChunk);
  uint64_t* const buf0 = Sm::spay();
  auto issue = [&](uint32_t c) {
    const uint64_t c0 = (uint64_t)c * kChunk;
    const uint32_t have = (uint32_t)min((uint64_t)kChunk, m - c0);
    const uint32_t bytes = ((have + 1) & ~1u) * 8u;
    const uint32_t g = gc + c, b = g % 3;
    mbar_expect_tx(Sm::cbar() + b, 2 * bytes);
    bulk_copy_g2s(buf0 + (size_t)b * 2 * kChunk, ska + c0, bytes, Sm::cbar() + b);
    bulk_copy_g2s(buf0 + (size_t)b * 2 * kChunk + kChunk, spa + c0, bytes, Sm::cbar() + b);
  };
  if(threadIdx.x == 0) { issue(0); if(nchunks > 1) issue(1); }
#pragma unroll 8
  for(uint32_t j = threadIdx.x; j < n; j += kThreads) atomicAdd(&tot[((uint32_t)sk[j] >> shift) & dmask], 1u);
  __syncthreads();
  {                                             // gbase = exclusive scan of the histogram
    uint32_t v = 0, inc = 0;
    if(threadIdx.x < kGsRadix) {
      v = tot[threadIdx.x]; inc = v;
#pragma unroll
      for(int s = 1; s < 32; s <<= 1) { const uint32_t o = __shfl_up_sync(MR_FULL_MASK, inc, s); if(lane >= (unsigned)s) inc += o; }
      if(lane == 31) Sm::wsum()[warp] = inc;
    }
    __syncthreads();
    if(threadIdx.x < kGsRadix) {
      uint32_t before = 0;
      for(unsigned w = 0; w < warp; ++w) before += Sm::wsum()[w];
      gbase[threadIdx.x] = before + inc - v;
      if(keep) { Sm::bsize()[threadIdx.x] = v; Sm::bstart()[threadIdx.x] = before + inc - v; }
    }
  }
  for(uint32_t c = 0; c < nchunks; ++c) {
    const uint32_t g = gc + c, b = g % 3;
    const uint64_t* kb = buf0 + (size_t)b * 2 * kChunk;
    const uint64_t* pb = kb + kChunk;
    uint16_t (*cnt)[kGsRadix] = C[c & 1];
    mbar_wait(Sm::cbar() + b, (g / 3) & 1u);
    uint64_t key[kFbRounds];
    uint32_t rk[kFbRounds];
    const uint64_t c0 = (uint64_t)c * kChunk;
    const uint32_t q0 = warp * (32 * kFbRounds) + lane;                   // this lane's first position inside the chunk
#pragma unroll
    for(int i = 0; i < kFbRounds; ++i) {
      const uint64_t pos = c0 + q0 + i * 32;
      const bool valid = pos >= skew && pos < m;
      key[i] = kb[q0 + i * 32];
      rk[i] = rank_round16(valid ? ((uint32_t)key[i] >> shift) & dmask : (uint32_t)kGsRadix, cnt[warp], lt);
    }
    __syncthreads();
    if(threadIdx.x == 0 && c + 2 < nchunks) issue(c + 2);                // its buffer was last read while chunk c - 1 was scattered
    if(threadIdx.x < kGsRadix) {
      uint32_t run = 0;
#pragma unroll 8
      for(int w = 0; w < kWarps; ++w) { const uint32_t t = cnt[w][threadIdx.x]; cnt[w][threadIdx.x] = (uint16_t)run; run += t; }
      const uint32_t at = gbase[threadIdx.x];
      cbase[threadIdx.x] = at; gbase[threadIdx.x] = at + run;
    }
    for(int i = threadIdx.x; i < kWarps * kGsRadix; i += kThreads) (&C[(c + 1) & 1][0][0])[i] = 0;
    __syncthreads();
#pragma unroll
    for(int i = 0; i < kFbRounds; ++i) {
      const uint64_t pos = c0 + q0 + i * 32;
      if(pos >= skew && pos < m) {
        const uint32_t d = ((uint32_t)key[i] >> shift) & dmask;
        const uint32_t dst = cbase[d] + cnt[warp][d] + rk[i];
        dk[dst] = key[i]; dp[dst] = pb[q0 + i * 32];
      }
    }
  }
  gc += nchunks;
  __syncthreads();
}

// ---- (3): (ak, ap)[0, n) sorted on key bits [0, bits) by LSD passes; the result is left in (ak, ap) when
// `stay`, else in (bk, bp) (the pass count is made even or odd accordingly); then the head bytes
template<int kThreads>
__device__ void sort_range_global(uint64_t* ak, uint64_t* ap, uint64_t* bk, uint64_t* bp, uint8_t* head,
                                  uint32_t n, int bits, bool stay, uint32_t& gc) {
  int passes = (bits + kGsDigit - 1) / kGsDigit;
  if(((passes & 1) == 0) != stay) ++passes;
  if(passes) {
    const int width = max(1, (bits + passes - 1) / passes);
    for(int p = 0; p < passes; ++p) {
      radix_pass_global<kThreads>(ak, ap, bk, bp, n, p * width, (1u << width) - 1, false, gc);
      uint64_t* t = ak; ak = bk; bk = t;
      t = ap; ap = bp; bp = t;
    }
  }
  // (ak, ap) hold the result; the writes are visible to the whole CTA (barrier at the end of the pass)
  for(uint32_t j = threadIdx.x; j < n; j += kThreads) head[j] = j == 0 || (uint32_t)ak[j] != (uint32_t)ak[j - 1];
  __syncthreads();
}

template<int kThreads>
__global__ void __launch_bounds__(kThreads, kThreads == 1024 ? 1 : 2) group_sort_kernel(group_sort_args A) {
  typedef gs_sm<kThreads> Sm;

  const uint32_t r = blockIdx.x;
  const uint64_t seg = A.hit_off[A.tile_first[r]];
  const uint64_t n64 = A.hit_off[A.tile_first[r + 1]] - seg;
  if(n64 == 0) return;
  const uint32_t n = (uint32_t)n64;
  const uint64_t rhi = (uint64_t)r << 32;
  uint32_t phase = 0, gc = 0;
  if(threadIdx.x == 0) { mbar_init(Sm::bar(), 1); mbar_init(Sm::cbar(), 1); mbar_init(Sm::cbar() + 1, 1); mbar_init(Sm::cbar() + 2, 1); }
  __syncthreads();
  uint64_t *kin = A.keys_in + seg, *pin = A.pays_in + seg, *ko = A.keys_out + seg, *po = A.pays_out + seg;
  uint8_t* head = A.head + seg;

  if(n <= A.cap) {
    sort_range_smem<kThreads>(kin, pin, ko, po, head, n, 0u, A.sr_bits, A.idx_bits, rhi, phase);
  } else {
    const int low_bits = A.sr_bits > kGsDigit ? A.sr_bits - kGsDigit : 0;
    if(low_bits + (int)A.range_idx_bits > 32) {
      sort_range_global<kThreads>(kin, pin, ko, po, head, n, A.sr_bits, false, gc);
    } else {
      // (2): cut by the top digit, then sort runs of consecutive buckets in shared memory
      radix_pass_global<kThreads>(kin, pin, ko, po, n, low_bits, kGsRadix - 1, true, gc);
      asm volatile("fence.proxy.async;" ::: "memory");        // the bulk copies below read what this CTA just stored
      __syncthreads();
      const uint32_t rcap = A.range_cap;
      uint32_t b = 0;
      while(b < (uint32_t)kGsRadix) {
        const uint32_t sz = Sm::bsize()[b];
        if(sz == 0) { ++b; continue; }
        const uint32_t at = Sm::bstart()[b];
        if(sz > rcap) {                                       // (3) on the bucket's low bits, back into place
          sort_range_global<kThreads>(ko + at, po + at, kin + at, pin + at, head + at, sz, low_bits, true, gc);
          asm volatile("fence.proxy.async;" ::: "memory");
          __syncthreads();
          ++b;
          continue;
        }
        uint32_t b1 = b + 1, total = sz;
        while(b1 < (uint32_t)kGsRadix) {
          const uint32_t nb = b1 + 1 - b;
          const int kb = low_bits + (32 - __clz(nb - 1));
          if(total + Sm::bsize()[b1] > rcap || kb + (int)A.range_idx_bits > 32) break;
          total += Sm::bsize()[b1];
          ++b1;
        }
        const uint32_t nb = b1 - b;
        const int kb = low_bits + (nb > 1 ? 32 - __clz(nb - 1) : 0);
        sort_range_smem<kThreads>(ko + at, po + at, ko + at, po + at, head + at, total, b << low_bits, kb, A.range_idx_bits, rhi, phase);
        b = b1;
      }
    }
  }
  // (every path ends with a barrier: the sorted slice is visible)
  if(threadIdx.x == 0 && (uint32_t)ko[n - 1] == A.nseq_all) atomicAdd(A.n_invalid_groups, 1ULL);
}

} // namespace

int group_sort_threads() {
  static const int v = [] { const char* e = getenv("MR_GSORT_THREADS"); const int x = e ? atoi(e) : 0; return x == 1024 ? 1024 : 512; }();
  return v;
}

// MR_GSORT_CAP lowers the capacity (a power of two, at least 32): the tests send the fixtures' reads through routes
// (2) and (3) that way
static int group_sort_cap_bits() {
  static const int env_bits = [] { const char* e = getenv("MR_GSORT_CAP"); int x = e ? atoi(e) : 0, b = 0; while((2 << b) <= x) ++b; return x >= 32 ? b : 31; }();
  return std::min(group_sort_threads() == 1024 ? 14 : 13, env_bits);
}

bool group_sort_usable(int sr_bits) {
  // route (2) needs 32-bit words for (low bits of the super-read index, position); beyond that every large read
  // would take route (3), and the device-wide radix sort does that job better
  return std::max(0, sr_bits - kGsDigit) + group_sort_cap_bits() <= 32;
}

int launch_group_sort(mr_context* ctx, group_sort_args A, uint32_t nreads) {
  if(!nreads) return MR_OK;
  const int cb = group_sort_cap_bits();
  A.range_idx_bits = (uint32_t)cb; A.range_cap = 1u << cb;
  A.idx_bits = (uint32_t)std::max(0, std::min(cb, 32 - A.sr_bits));
  A.cap = A.sr_bits + 5 <= 32 ? 1u << A.idx_bits : 0u;        // whole reads in shared memory: up to this many hits
  typedef void (*kernel_t)(group_sort_args);
  const bool wide = group_sort_threads() == 1024;
  const kernel_t fn = wide ? group_sort_kernel<1024> : group_sort_kernel<512>;
  const size_t smem = wide ? gs_layout<1024>::bytes : gs_layout<512>::bytes;
  MR_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fn<<<nreads, wide ? 1024 : 512, smem, ctx->stream>>>(A);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

// Device-resident super-read index: 2-bit text, suffix array, per-entry k-mer tails, prefix
// counts and the tables that map a text position to (super-read, offset).
//
// Layout in HBM (n = text bases, m = psa-min, k = mer, nsa = n - m + 1):
//   text   uint64[ceil(n/32)+2]  reference compact_dna layout (base i at bits 2(i%32)), zero padded
//   sa     uint32[nsa]           positions ordered by (k-mer padded with A, position descending)
//                                == the order of SA::sort_one_mer (mer_sa_imp.hpp:352-366)
//   tails  u8/u16/u32[nsa]       low 2(k-mi) bits of each entry's padded k-mer: a lookup never
//                                touches the text, one probe is one small read next to its
//                                neighbours instead of the reference's SA read + text read
//   counts uint32[4^mi+1]        exclusive prefix of the mi-mer histogram (mer_sa_imp.hpp:317-330).
//                                mi <= m is an INTERNAL prefix length, chosen so that counts + tails
//                                are of the order of the 126 MB L2 when the index is small enough
//                                (C2: mi = 12, 67 MB + 36 MB) while buckets stay short; the
//                                (index, nb) a lookup returns does not depend on it.  The reference's 4^m + 1 table is
//                                recomputed on demand for the parity tap (mr_index_export_counts).
//   sr_start uint32[nseq+1], blk uint32[(n>>8)+2]: blk[b] = sequence containing base b*256
//
// Texts of 2^32 bases or more (BASELINE configs[3], human-size): the super-reads are cut, at
// super-read boundaries, into up to kMaxParts PARTS of fewer than 2^32 bases; every part is a
// complete index of the kind above over its own text (positions, ranks and counts stay 32 bit, the
// lookup kernels are the same) and a k-mer's list is the concatenation of its per-part lists.
// What makes that identical to one suffix array over the whole text:
//   * a super-read lies in exactly one part and the order of a part's suffix array restricted to
//     one super-read is the order of the global one (same keys, positions shifted by a constant),
//     so every (read, super-read, strand) hit list comes out in the reference's order;
//   * the list size the count filters see (coarse_aligner.cc:108-125) is the sum over the parts.
//     The global suffix array also matches k-mers that straddle two consecutive super-reads (they
//     count, and are dropped later by pos_iterator): a part's text is therefore extended by the
//     first k-1 bases of the next part, so these positions keep their k-mer; the extension's own
//     positions are suffixes shorter than k inside the part, which never match, and are counted by
//     the next part, where they are ordinary positions.
#pragma once
#include "common.cuh"
#include <vector>

constexpr int kBlkShift  = 8;
constexpr int kMaxShort  = 16;    // k - m <= 16 (tails are 32 bit)
constexpr int kMaxParts  = 4;     // parts of one index (texts up to ~2^34 bases)

struct index_view {
  const uint32_t* __restrict__ counts;
  const void*     __restrict__ tails;
  const uint32_t* __restrict__ sa;
  const uint32_t* __restrict__ sr_start;
  const uint32_t* __restrict__ blk;
  const uint4*    __restrict__ blkx;   // blkx[b] = { blk[b], sr_start[blk[b]], sr_start[blk[b] + 1], 0 }: one load locates a hit
  uint64_t n;
  uint32_t nsa, nseq, k, m, mi, tail_bits, tail_bytes, nshort;
  // Compact form of `counts` for the lookups (null when the buckets are too large for it to pay):
  // the sizes of 32 consecutive buckets as 4-bit numbers in one 16-byte record plus the start of the
  // group's first bucket in gbase[]; a bucket's bounds are gbase + a sum of nibbles (two multiplies).
  // 5 bits per prefix instead of 32: with the 8-bit tails, what a lookup reads at random shrinks from
  // 103 MB to 47 MB on the yeast-size index and stays in the L2 (ncu: sector hit rate 41 % -> 90 %, DRAM
  // bytes per launch 4.4 GB -> 0.4 GB).  A group with a bucket of 15 entries or more has nibble 0 = 15
  // and is looked up in `counts` as before.
  const ulonglong2* __restrict__ nib;    // one record per group of 32 prefixes
  const uint32_t*   __restrict__ gbase;
  // saloc[i] = (super-read, 1-based offset) of suffix-array entry i for a mer of k bases, or (0xffffffff, 0) when the
  // k-mer there crosses into the next sequence (pos_iterator, superread_parser.hpp:110-134, done once at build time):
  // expanding a hit is one 8-byte read next to its list neighbours instead of a 4-byte read plus a dependent random
  // 16-byte one into the block table.
  const uint2*      __restrict__ saloc;
  uint32_t own;                    // bases of the part's own super-reads (sr_start[nseq]); n - own = extension (index.cuh header)
  uint32_t sr_base;                // global index of this part's first super-read (0 for a one-part index)
  uint32_t nseq_all;               // super-reads of the whole index (== nseq for a one-part index)
  uint64_t short_key[kMaxShort];   // padded k-mers of the tail-short suffixes (positions n-k+1 .. n-m)
};

struct mr_index {
  mr_context* ctx = nullptr;
  uint64_t n = 0;
  uint32_t nsa = 0, nseq = 0, k = 0, m = 0, mi = 0, n_unitigs = 0;
  bool     has_unitigs = false;
  bool     unitig_ids_ok = true;     // every id of the unitig paths is below n_unitigs (the overlap graph and the
                                     // printing index unitig_len with them unchecked, as the reference does)
  uint64_t unitig_total = 0;         // entries of unitig_ids
  uint64_t inputs_checksum = 0;      // mr_inputs_checksum of what the index was built from
  dev_buf  text, sa, tails, counts, sr_start, blk;
  dev_buf  nib, gbase;               // see index_view::nib (derived; not in index files)
  dev_buf  saloc;                    // see index_view::saloc (derived; not in index files)
  dev_buf  blkx;                     // uint4[(n>>8)+1]: see index_view::blkx (derived; not in index files)
  dev_buf  lut;                      // counts and tails live side by side in this one allocation
  int alloc_lut(mr_context* c, size_t counts_bytes, size_t tails_bytes) {
    const size_t off = (counts_bytes + 255) & ~(size_t)255;
    const int rc = lut.ensure(c, off + tails_bytes);
    if(rc != MR_OK) return rc;
    counts.alias(lut.p, counts_bytes);
    tails.alias((char*)lut.p + off, tails_bytes);
    lut_bytes = off + tails_bytes;
    return MR_OK;
  }
  size_t   lut_bytes = 0;
  uint64_t nib_overflow_groups = 0;  // groups of 64 prefixes that hold a bucket of 15 or more entries (looked up in counts)
  dev_buf  unitig_ids, unitig_off, unitig_len, sr_nunitigs;
  index_view view;
  // whole-index tables (a one-part index: the part is the index itself)
  uint64_t n_all = 0;                // bases of all super-reads
  uint32_t nseq_all = 0;             // number of super-reads
  dev_buf  sr_len;                   // uint32[nseq_all]: length of every super-read, by global index
  std::vector<mr_index*> more;       // parts 1 .. P-1 (owned); part 0 is this object
  dev_buf  more_views;               // index_view[P-1] on the device, for the kernels that walk the parts
  uint32_t nparts() const { return 1 + (uint32_t)more.size(); }
  const index_view& part_view(uint32_t p) const { return p == 0 ? view : more[p - 1]->view; }
  ~mr_index() { for(mr_index* m_ : more) delete m_; }
};

// counts[p], counts[p + 1] with one 16-byte load (plus a 4-byte one when p % 4 == 3): the two
// entries almost always share a 32-byte sector, and a random sector fetched once must not be
// requested a second time by a separate load instruction after it has left the L1.
__device__ __forceinline__ void load_count_pair(const uint32_t* __restrict__ counts, uint32_t p, uint32_t& c0, uint32_t& c1) {
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(counts) + (p >> 2));
  switch(p & 3) {
  case 0: c0 = v.x; c1 = v.y; break;
  case 1: c0 = v.y; c1 = v.z; break;
  case 2: c0 = v.z; c1 = v.w; break;
  default: c0 = v.w; c1 = __ldg(counts + p + 1);
  }
}

// sum of the sixteen 4-bit fields of x (each at most 14 where it matters: the total stays below 256)
__device__ __forceinline__ uint32_t nibble_sum(uint64_t x) {
  const uint64_t t = (x & 0x0f0f0f0f0f0f0f0fULL) + ((x >> 4) & 0x0f0f0f0f0f0f0f0fULL);
  return (uint32_t)((t * 0x0101010101010101ULL) >> 56);
}
// bounds [c0, c1) of the bucket of prefix p: from the nibble record when the index has one (kNib), else counts[p], counts[p + 1]
template<bool kNib>
__device__ __forceinline__ void bucket_bounds(const index_view& iv, uint32_t p, uint32_t& c0, uint32_t& c1) {
  if(kNib) {
    const uint32_t g = p >> 5, j = p & 31;
    const ulonglong2 rec = __ldg(iv.nib + g);
    const uint32_t base = __ldg(iv.gbase + g);           // issued with the record, not after a look at it
    if((rec.x & 15ULL) != 15ULL) {
      const uint64_t w = j < 16 ? rec.x : rec.y;
      const uint32_t sh = 4 * (j & 15);
      const uint32_t before = nibble_sum(w & ((1ULL << sh) - 1)) + (j < 16 ? 0u : nibble_sum(rec.x));
      c0 = base + before;
      c1 = c0 + (uint32_t)((w >> sh) & 15ULL);
      return;
    }
  }
  load_count_pair(iv.counts, p, c0, c1);
}

__device__ __forceinline__ uint32_t load_tail(const index_view& iv, uint32_t i) {
  if(iv.tail_bytes == 1) return __ldg(reinterpret_cast<const uint8_t*>(iv.tails) + i);
  if(iv.tail_bytes == 2) return __ldg(reinterpret_cast<const uint16_t*>(iv.tails) + i);
  return __ldg(reinterpret_cast<const uint32_t*>(iv.tails) + i);
}

// ---- bucket search ---------------------------------------------------------------------------
// tails are read as aligned 32-bit words (4 / 2 / 1 entries each) and compared with the per-byte /
// per-halfword SIMD instructions: a bucket of 8 one-byte tails costs 2-3 loads and ~25 instructions
// instead of 8 loads and ~80.
__device__ __forceinline__ uint32_t tail_word(const index_view& iv, uint32_t word_index) {
  return __ldg(reinterpret_cast<const uint32_t*>(iv.tails) + word_index);
}
__device__ __forceinline__ uint32_t tail_word_of(const index_view& iv, uint32_t entry) {   // word holding `entry`
  return iv.tail_bytes == 1 ? entry >> 2 : (iv.tail_bytes == 2 ? entry >> 1 : entry);
}

// entries of tails[a0, a1) that are < t (less) and <= t (leq); w0 = the word holding entry a0, already loaded
__device__ __forceinline__ void bucket_count(const index_view& iv, uint32_t a0, uint32_t a1, uint32_t t, uint32_t w0,
                                             uint32_t& less, uint32_t& leq) {
  less = 0; leq = 0;
  if(iv.tail_bytes == 4) {
    less = w0 < t; leq = w0 <= t;
    for(uint32_t i = a0 + 1; i < a1; ++i) { const uint32_t v = tail_word(iv, i); less += v < t; leq += v <= t; }
    return;
  }
  const bool bytes = iv.tail_bytes == 1;
  const uint32_t epw_shift = bytes ? 2 : 1, ebits = bytes ? 8 : 16;
  const uint32_t trep = bytes ? t * 0x01010101u : t * 0x00010001u;
  uint32_t w = w0;
  for(uint32_t base = a0 & ~((1u << epw_shift) - 1); base < a1; base += 1u << epw_shift) {
    if(base > a0) w = tail_word(iv, base >> epw_shift);
    const uint32_t skip = base < a0 ? a0 - base : 0;                         // entries of this word before the bucket
    const uint32_t have = min(1u << epw_shift, a1 - base);                   // entries of this word inside [.., a1)
    const uint32_t hi = have == (1u << epw_shift) ? 0xffffffffu : ((1u << (ebits * have)) - 1);
    const uint32_t vmask = hi & ~((1u << (ebits * skip)) - 1);
    const uint32_t lt = (bytes ? __vcmpltu4(w, trep) : __vcmpltu2(w, trep)) & vmask;
    const uint32_t le = (bytes ? __vcmpleu4(w, trep) : __vcmpleu2(w, trep)) & vmask;
    less += __popc(lt) >> (bytes ? 3 : 4);
    leq  += __popc(le) >> (bytes ? 3 : 4);
  }
}

// [lo, hi) of tails[a0, a1) equal to t
__device__ __forceinline__ void bucket_range(const index_view& iv, uint32_t a0, uint32_t a1, uint32_t t, uint32_t w0,
                                             uint32_t& lo, uint32_t& hi) {
  if(a1 - a0 <= 64) {
    uint32_t less, leq;
    bucket_count(iv, a0, a1, t, w0, less, leq);
    lo = a0 + less; hi = a0 + leq;
  } else {
    uint32_t a = a0, b = a1;
    while(a < b) { const uint32_t mid = a + ((b - a) >> 1); if(load_tail(iv, mid) < t) a = mid + 1; else b = mid; }
    lo = a; b = a1;
    while(a < b) { const uint32_t mid = a + ((b - a) >> 1); if(load_tail(iv, mid) <= t) a = mid + 1; else b = mid; }
    hi = a;
  }
}

// bucket_range for one-byte tails (k - mi <= 4: the production mer lengths), without the width dispatch
__device__ __forceinline__ void bucket_range_bytes(const index_view& iv, uint32_t a0, uint32_t a1, uint32_t t, uint32_t w0,
                                                   uint32_t& lo, uint32_t& hi) {
  if(a1 - a0 > 64) { bucket_range(iv, a0, a1, t, w0, lo, hi); return; }
  const uint32_t trep = t * 0x01010101u;
  const uint32_t* words = reinterpret_cast<const uint32_t*>(iv.tails);
  uint32_t less = 0, leq = 0, w = w0;
  for(uint32_t base = a0 & ~3u; base < a1; base += 4) {
    if(base > a0) w = __ldg(words + (base >> 2));
    const uint32_t skip = base < a0 ? a0 - base : 0;
    const uint32_t have = min(4u, a1 - base);
    const uint32_t vmask = (have == 4 ? 0xffffffffu : ((1u << (8 * have)) - 1)) & ~((1u << (8 * skip)) - 1);
    less += __popc(__vcmpltu4(w, trep) & vmask) >> 3;
    leq  += __popc(__vcmpleu4(w, trep) & vmask) >> 3;
  }
  lo = a0 + less; hi = a0 + leq;
}

// [index, nb) of SA entries whose text equals `mer` (mer_sa_imp.hpp:369-479 returns the same pair)
__device__ __forceinline__ void index_lookup(const index_view& iv, uint64_t mer, uint32_t& index, uint32_t& nb) {
  const uint32_t pre = (uint32_t)(mer >> iv.tail_bits);
  const uint32_t t   = (uint32_t)mer & (iv.tail_bits >= 32 ? 0xffffffffu : ((1u << iv.tail_bits) - 1));
  uint32_t c0, c1;
  if(iv.nib) bucket_bounds<true>(iv, pre, c0, c1); else load_count_pair(iv.counts, pre, c0, c1);
  index = 0; nb = 0;
  if(c0 == c1) return;
  uint32_t lo, hi;
  bucket_range(iv, c0, c1, t, tail_word(iv, tail_word_of(iv, c0)), lo, hi);
  if(hi == lo) return;
  // Suffixes shorter than k sort first inside their padded-equal range (larger position first)
  // and never match (mer_sa_imp.hpp:399-406).  Only k-mers ending in A can collide with them.
  if((mer & 3) == 0) {
    for(uint32_t j = 0; j < iv.nshort; ++j) lo += iv.short_key[j] == mer;
  }
  nb = hi - lo;
  index = nb ? lo : 0;
}

// The same for a pattern of kk <= k bases (the fine pass looks shorter mers up in the same suffix
// array; mer_sa_imp.hpp:376-381 when kk <= psa-min, :382-479 otherwise): the entries whose text
// STARTS with the pattern.  They are the padded k-mers in [mer << s, ((mer + 1) << s) - 1],
// s = 2 (k - kk); suffixes with fewer than kk bases left carry the smallest key of that range
// (their missing bases are padded with A) and never match.
__device__ __forceinline__ void index_lookup_prefix(const index_view& iv, uint64_t mer, uint32_t kk, uint32_t& index, uint32_t& nb) {
  const uint32_t s = 2 * (iv.k - kk);
  uint32_t lo, hi;
  if(kk <= iv.mi) {
    const uint32_t sh = 2 * (iv.mi - kk);
    lo = __ldg(iv.counts + (uint32_t)(mer << sh));
    hi = __ldg(iv.counts + (uint32_t)((mer + 1) << sh));
  } else {
    const uint32_t rb = 2 * (kk - iv.mi);                       // pattern bits below the table prefix
    const uint32_t pre = (uint32_t)(mer >> rb);
    const uint32_t t_lo = (uint32_t)((mer & ((1ULL << rb) - 1)) << s);
    const uint32_t t_hi = t_lo | (s ? ((1u << s) - 1) : 0u);
    uint32_t c0, c1;
    load_count_pair(iv.counts, pre, c0, c1);
    lo = hi = c0;
    if(c0 != c1) {
      if(c1 - c0 <= 64) {
        const uint32_t w0 = tail_word(iv, tail_word_of(iv, c0));
        uint32_t less, leq, dummy;
        bucket_count(iv, c0, c1, t_lo, w0, less, dummy);
        bucket_count(iv, c0, c1, t_hi, w0, dummy, leq);
        lo = c0 + less; hi = c0 + leq;
      } else {
        uint32_t a = c0, b = c1;
        while(a < b) { const uint32_t mid = a + ((b - a) >> 1); if(load_tail(iv, mid) < t_lo) a = mid + 1; else b = mid; }
        lo = a; b = c1;
        while(a < b) { const uint32_t mid = a + ((b - a) >> 1); if(load_tail(iv, mid) <= t_hi) a = mid + 1; else b = mid; }
        hi = a;
      }
    }
  }
  if(hi != lo) {
    for(uint32_t j = 0; j < iv.nshort; ++j)                     // short_key[j]: the suffix with k - 1 - j bases
      lo += (iv.k - 1 - j < kk) && (iv.short_key[j] >> s) == mer;
  }
  nb = hi - lo;
  index = nb ? lo : 0;
}

// SA entry x -> (super-read, 1-based offset) for a mer of kk bases; false when it crosses into the next sequence
__device__ __forceinline__ bool index_locate_k(const index_view& iv, uint32_t x, uint32_t kk, uint32_t& sr, uint32_t& off) {
  if(x >= iv.own) return false;              // a position of the extension: it belongs to the next part
  const uint4 b = __ldg(iv.blkx + (x >> kBlkShift));
  uint32_t i = b.x, s0 = b.y, s1 = b.z;
  while(s1 <= x) { ++i; s0 = s1; s1 = __ldg(iv.sr_start + i + 1); }
  if((uint64_t)x + kk > s1) return false;
  sr  = i;
  off = x - s0 + 1;
  return true;
}

// SA entry x -> (super-read, 1-based offset); false when x + k crosses into the next sequence
// (pos_iterator::operator++, superread_parser.hpp:110-134)
__device__ __forceinline__ bool index_locate(const index_view& iv, uint32_t x, uint32_t& sr, uint32_t& off) {
  const uint4 b = __ldg(iv.blkx + (x >> kBlkShift));     // sequence of the block's first base and its bounds
  uint32_t i = b.x, s0 = b.y, s1 = b.z;
  while(s1 <= x) { ++i; s0 = s1; s1 = __ldg(iv.sr_start + i + 1); }
  if((uint64_t)x + iv.k > s1) return false;
  sr  = i;
  off = x - s0 + 1;
  return true;
}

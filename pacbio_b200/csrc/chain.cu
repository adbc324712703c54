// Chaining ("LIS") + coords: one warp per (read, super-read) group.
//   chain_*        == lis_align::compute_L_P (lis_align.hpp:139-182), window_size 1
//   finish_group   == compute_coords_info + least_square_2d + canonicalize + the filters of
//                     align_sequence_max (pb_aligner.cc:11-82, least_square_2d.hpp:47-67,
//                     pb_aligner.hpp:151-174, coarse_aligner.cc:42-60)
//
// The reference walks a forward_list L for every new hit, stops at the first feasible extension and
// inserts the new element after the first strict minimum of `len` seen on the way.  Here L is an
// array kept in REVERSE list order (list front == array end): 32 entries are tested per step, a
// ballot finds the first feasible one, a redux finds the insertion point, and the usual case --
// extend the newest chain, insert at the front -- touches only the last array slots.
//
// Groups are binned by size: <= 64 hits and <= 1024 hits keep L, the chain-start coordinates and
// the back pointers in shared memory (22 B per hit); larger groups run the same algorithm out of
// global scratch.  The kernels are latency/issue bound, not bandwidth bound: what matters is the
// length of the dependent chain per hit (one shared-memory round trip + ~10 FP64 ops + 3 warp
// collectives) and the number of warps in flight.
#include "align.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <string>
#include <vector>

namespace {

constexpr uint32_t kThreadFinishLongMax = 1536;   // chains up to this many hits: one thread each; longer: one warp each

// (C < 0 / a < 0: lis_align::accept_all, the predicates of the fine pass, fine_aligner.cc:43-46)
// Tried and dropped: an integer form of both predicates (d1 <= floor(b + a d2) as a multiply-shift whose multiplier the
// host verifies against the FP64 table for every d up to the cap).  Exact, but the chaining kernels are bound by their
// shared-memory round trips and warp collectives, not by these ten FP64 instructions: 26.1 against 25.7 ms per step.
__device__ __forceinline__ bool accept_mer(int32_t pb_i, int32_t sr_i, int32_t lpb, int32_t lsr, double a, double b, double C) {
  if(C < 0.0) return true;
  const double d1 = (double)(pb_i - lpb), d2 = (double)(sr_i - lsr);
  const double t1 = a * d2, t2 = a * d1;                   // mul then add, never fused (-fmad=false)
  return d1 <= b + t1 && d2 <= b + t2 && d1 <= C && d2 <= C;
}

__device__ __forceinline__ bool accept_sequence(int32_t span_pb, int32_t span_sr, double a) {
  if(a < 0.0) return true;
  const double s1 = a * (double)span_sr, s2 = a * (double)span_pb;
  return (double)span_pb <= s1 && (double)span_sr <= s2;
}

// x / n for an integer count n given r = RN(1/n): q = RN(x*r) is within one ulp of x/n, the
// remainder x - q*n is exact in one FMA, and q + rem*r rounds to the correctly rounded quotient
// (Markstein's division theorem) -- bit-identical to the IEEE division the reference executes,
// at 3 FP64 instructions instead of a ~35-instruction division sequence.  The online least
// squares divides four values by the same n for every chain element.
__device__ __forceinline__ double div_by_count(double x, double dn, double r) {
  const double q = x * r;
  const double rem = __fma_rn(-q, dn, x);
  return __fma_rn(rem, r, q);
}

// RN(1 / n) for the chain lengths one thread handles: the count is the same in every lane, so this
// is one broadcast read from the constant cache instead of a ~40-instruction IEEE division per element
constexpr uint32_t kRcpMax = 2048;
__constant__ double kRcpTable[kRcpMax + 1];
__device__ __forceinline__ double rcp_count(uint32_t n) { return n <= kRcpMax ? kRcpTable[n] : 1.0 / (double)n; }

// ---------------------------------------------------------------------------------------------
// shared-memory strand: per warp arrays of CAP entries
// ---------------------------------------------------------------------------------------------
// One group's working set, carved out of the block's dynamic shared memory: `cap` entries per
// array, 22 B per hit in all (cap is a multiple of 64).
struct warp_store {
  int32_t  *pb, *sr, *cpb, *csr;
  uint32_t *meta;              // len << 16 | element index   (cap <= 65536)
  uint16_t *pprev;             // by element index, 0xffff = none
  __device__ __forceinline__ warp_store(unsigned char* base, uint32_t cap) {
    pb = reinterpret_cast<int32_t*>(base); sr = pb + cap; cpb = sr + cap; csr = cpb + cap;
    meta = reinterpret_cast<uint32_t*>(csr + cap);
    pprev = reinterpret_cast<uint16_t*>(meta + cap);
  }
};
__host__ __device__ constexpr size_t warp_store_bytes(uint32_t cap, bool taps) {
  return (size_t)cap * 22 + (taps ? (size_t)cap * 2 : 0);
}

template<bool TAPS>
__device__ __forceinline__ void chain_strand_smem(const uint64_t* __restrict__ pay, uint32_t N, bool neg, const warp_store& S,
                                                  uint16_t* sub, double a, double b, double C,
                                                  uint32_t& longest_out, uint32_t& best_out) {
  const unsigned lane = threadIdx.x & 31;
  const unsigned lt = lanemask_lt();
  uint32_t cnt = 0, longest = 0, best = 0, nsub = 0;
  int32_t  fr_pb = 0, fr_sr = 0, fr_cpb = 0, fr_csr = 0;    // list front (array slot cnt - 1), same in every lane
  uint32_t fr_meta = 0;
  uint64_t next_pl = lane < N ? pay[lane] : 0;
  for(uint32_t base = 0; base < N; base += 32) {
    const uint32_t il = base + lane;
    const uint64_t pl = next_pl;
    if(base + 32 < N) next_pl = (il + 32 < N) ? pay[il + 32] : 0;      // prefetch the next 32 hits
    const int32_t pb_l = (int32_t)(uint32_t)pl, sr_l = (int32_t)(uint32_t)(pl >> 32);
    const bool mine = il < N && ((sr_l < 0) == neg);
    const unsigned mine_mask = __ballot_sync(MR_FULL_MASK, mine);
    if(!mine_mask) continue;
    // 32 hits at once: does each hit extend the hit just before it (same strand)?  Whenever that
    // earlier hit sits at the list front when its successor is processed, the reference's walk stops
    // on it immediately, so whole runs of such hits are appended in one step below.
    const unsigned below = mine_mask & lt;
    const int pred_lane = below ? 31 - __clz(below) : 0;
    const int32_t ppb = __shfl_sync(MR_FULL_MASK, pb_l, pred_lane), psr = __shfl_sync(MR_FULL_MASK, sr_l, pred_lane);
    const bool ext = mine && below && sr_l > psr && accept_mer(pb_l, sr_l, ppb, psr, a, b, C);
    const unsigned ext_mask = __ballot_sync(MR_FULL_MASK, ext);
    unsigned todo = mine_mask;
    while(todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t i = base + src;
      const int32_t pb_i = __shfl_sync(MR_FULL_MASK, pb_l, src), sr_i = __shfl_sync(MR_FULL_MASK, sr_l, src);
      if(TAPS) { if(lane == 0) sub[i] = (uint16_t)nsub; }
      ++nsub;

      int      found = -1, prev_pos = -1;
      uint32_t f_meta = 0, min_len = 0xffffffffu;
      int32_t  f_cpb = 0, f_csr = 0;
      // Fast path: the list front (kept in registers) is feasible: the walk stops at position 0
      // without passing any entry, so the new element goes to the front.
      if(cnt != 0 && sr_i > fr_sr && accept_mer(pb_i, sr_i, fr_pb, fr_sr, a, b, C)) {
        found = 0; f_meta = fr_meta; f_cpb = fr_cpb; f_csr = fr_csr;
      } else
      for(uint32_t c0 = 0; c0 < cnt; c0 += 32) {
        const uint32_t p = c0 + lane;
        const bool in = p < cnt;
        const uint32_t slot = cnt - 1 - p;
        int32_t lsr = 0, lpb = 0; uint32_t meta = 0;
        if(in) { lsr = S.sr[slot]; lpb = S.pb[slot]; meta = S.meta[slot]; }
        const bool feas = in && sr_i > lsr && accept_mer(pb_i, sr_i, lpb, lsr, a, b, C);
        const unsigned ball = __ballot_sync(MR_FULL_MASK, feas);
        const unsigned limit = ball ? (unsigned)(__ffs(ball) - 1) : 32u;
        // first position of the strict minimum of len among the entries walked over
        const unsigned packed = (in && lane < limit) ? (((meta >> 16) << 5) | lane) : 0xffffffffu;
        const unsigned bp = __reduce_min_sync(MR_FULL_MASK, packed);
        if(bp != 0xffffffffu && (bp >> 5) < min_len) { min_len = bp >> 5; prev_pos = (int)(c0 + (bp & 31)); }
        if(ball) {
          found = (int)(c0 + limit);
          f_meta = __shfl_sync(MR_FULL_MASK, meta, limit);
          const uint32_t fslot = cnt - 1 - (uint32_t)found;
          f_cpb = S.cpb[fslot]; f_csr = S.csr[fslot];           // uniform address: broadcast
          break;
        }
      }
      const uint32_t e_len = found >= 0 ? (f_meta >> 16) + 1 : 1;
      const int32_t cpb = found >= 0 ? f_cpb : pb_i, csr = found >= 0 ? f_csr : sr_i;
      // insert after prev_pos: the q = prev_pos + 1 entries in front of it move up one slot
      const uint32_t q = (uint32_t)(prev_pos + 1);
      for(uint32_t top = cnt; top > cnt - q; ) {
        const uint32_t lo = (top - (cnt - q)) > 32 ? top - 32 : cnt - q;
        const uint32_t s = lo + lane;
        const bool has = s < top;
        int32_t v0 = 0, v1 = 0, v2 = 0, v3 = 0; uint32_t v4 = 0;
        if(has) { v0 = S.pb[s]; v1 = S.sr[s]; v2 = S.cpb[s]; v3 = S.csr[s]; v4 = S.meta[s]; }
        __syncwarp();
        if(has) { S.pb[s + 1] = v0; S.sr[s + 1] = v1; S.cpb[s + 1] = v2; S.csr[s + 1] = v3; S.meta[s + 1] = v4; }
        __syncwarp();
        top = lo;
      }
      if(lane == 0) {
        const uint32_t s = cnt - q;
        S.pb[s] = pb_i; S.sr[s] = sr_i; S.cpb[s] = cpb; S.csr[s] = csr; S.meta[s] = (e_len << 16) | i;
        S.pprev[i] = found >= 0 ? (uint16_t)(f_meta & 0xffff) : (uint16_t)0xffff;
      }
      ++cnt;
      if(longest < e_len && accept_sequence(pb_i - cpb, sr_i - csr, a)) { longest = e_len; best = i; }
      if(q == 0) { fr_pb = pb_i; fr_sr = sr_i; fr_cpb = cpb; fr_csr = csr; fr_meta = (e_len << 16) | i; }
      else if(q > 32) { __syncwarp(); continue; }   // deep in the list: its successors take the normal route

      // Run: the hits right after this one that each extend their predecessor.  When such a hit is
      // processed its predecessor sits at list position q, so its walk passes the same q entries this
      // one passed: if none of them is feasible for it, the walk stops on the predecessor and the first
      // strict minimum of len over those q entries is again entry q - 1 -- the hit lands at position q
      // too, in front of its predecessor.  The whole run is appended in one step: lane t of the run gets
      // len + 1 + t, the same chain start, its predecessor as back pointer.  (q == 0, nothing in
      // front, is the common case; q > 0 happens when an early stray hit with a large super-read
      // offset stays at the list front and every hit of the real alignment files in behind it.)
      const unsigned stop_mask = todo & ~ext_mask;
      unsigned run = stop_mask ? (todo & ((1u << (__ffs(stop_mask) - 1)) - 1)) : todo;
      if(run && q != 0) {
        __syncwarp();
        bool blocked = false;
        if((run >> lane) & 1) {
          for(uint32_t p = 0; p < q; ++p) {
            const uint32_t slot = cnt - 1 - p;
            const int32_t lsr = S.sr[slot], lpb = S.pb[slot];
            blocked |= sr_l > lsr && accept_mer(pb_l, sr_l, lpb, lsr, a, b, C);
          }
        }
        const unsigned bm = __ballot_sync(MR_FULL_MASK, blocked);
        if(bm) run &= (1u << (__ffs(bm) - 1)) - 1;
        if(run) {                                   // the q entries in front move up by the run's length
          const uint32_t r = __popc(run), s = cnt - q + lane;
          const bool has = lane < q;
          int32_t v0 = 0, v1 = 0, v2 = 0, v3 = 0; uint32_t v4 = 0;
          if(has) { v0 = S.pb[s]; v1 = S.sr[s]; v2 = S.cpb[s]; v3 = S.csr[s]; v4 = S.meta[s]; }
          __syncwarp();
          if(has) { S.pb[s + r] = v0; S.sr[s + r] = v1; S.cpb[s + r] = v2; S.csr[s + r] = v3; S.meta[s + r] = v4; }
        }
      }
      if(run) {
        const uint32_t r = __popc(run);
        const bool inrun = (run >> lane) & 1;
        const uint32_t t = __popc(run & lt);
        const uint32_t my_len = e_len + 1 + t;
        if(inrun) {
          const uint32_t s = cnt - q + t;
          S.pb[s] = pb_l; S.sr[s] = sr_l; S.cpb[s] = cpb; S.csr[s] = csr; S.meta[s] = (my_len << 16) | il;
          S.pprev[il] = (uint16_t)(base + pred_lane);
          if(TAPS) sub[il] = (uint16_t)(nsub + t);
        }
        // `longest` only moves up and len grows along the run: the last accepted element wins
        const bool acc = inrun && my_len > longest && accept_sequence(pb_l - cpb, sr_l - csr, a);
        const unsigned accm = __ballot_sync(MR_FULL_MASK, acc);
        if(accm) {
          const int hl = 31 - __clz(accm);
          longest = e_len + 1 + __popc(run & ((1u << hl) - 1));
          best = base + hl;
        }
        if(q == 0) {
          const int last = 31 - __clz(run);
          fr_pb = __shfl_sync(MR_FULL_MASK, pb_l, last); fr_sr = __shfl_sync(MR_FULL_MASK, sr_l, last);
          fr_meta = ((e_len + r) << 16) | (base + last);
        }
        cnt += r; nsub += r; todo &= ~run;
      }
      __syncwarp();
    }
  }
  longest_out = longest;
  best_out = best;
}

// ---------------------------------------------------------------------------------------------
// global-memory strand (groups larger than the shared-memory tiers)
// ---------------------------------------------------------------------------------------------
// window > 1 (--window-size, lis_align.hpp:17-45,162-163): the mer predicate applies to the sum of the last `window`
// steps of a chain and only once the chain has that many.  That sum is X[i] - X[w], w the element `window` steps
// back from i -- the (window-1)-th ancestor of the list element the new hit would extend -- so a list entry
// carries the coordinates of that ancestor (Lwpb / Lwsr; kNoWindow while its chain is too short to be tested)
// next to its own, which the increasing test still uses.  The shared-memory kernels implement window 1 only;
// with a larger window every group comes here.
constexpr int32_t kNoWindow = (int32_t)0x80000000;
__device__ void chain_strand_global(const uint64_t* __restrict__ pay, uint32_t N, bool neg, const chain_buffers& cb, uint64_t gs,
                                    double a, double b, double C, uint32_t& longest_out, uint32_t& best_out, uint32_t* tap_sub,
                                    const uint8_t* removed = nullptr, uint32_t window = 1) {
  const unsigned lane = threadIdx.x & 31;
  const bool win = window > 1;
  int32_t*  Lwpb = win ? cb.Lwpb + gs : nullptr; int32_t* Lwsr = win ? cb.Lwsr + gs : nullptr;
  int32_t*  Lpb  = cb.Lpb + gs;  int32_t* Lsr = cb.Lsr + gs;
  uint32_t* Llen = cb.Llen + gs; uint32_t* Lelt = cb.Lelt + gs;
  uint32_t* pprev = cb.pprev + gs; uint32_t* cstart = cb.cstart + gs;
  uint32_t cnt = 0, longest = 0, best = 0, nsub = 0;
  for(uint32_t base = 0; base < N; base += 32) {
    const uint32_t il = base + lane;
    const uint64_t pl = il < N ? pay[il] : 0;
    const int32_t pb_l = (int32_t)(uint32_t)pl, sr_l = (int32_t)(uint32_t)(pl >> 32);
    unsigned todo = __ballot_sync(MR_FULL_MASK, il < N && ((sr_l < 0) == neg) && !(removed && removed[il]));
    while(todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t i = base + src;
      const int32_t pb_i = __shfl_sync(MR_FULL_MASK, pb_l, src), sr_i = __shfl_sync(MR_FULL_MASK, sr_l, src);
      if(tap_sub && lane == 0) tap_sub[gs + i] = nsub;
      ++nsub;
      int      found = -1, prev_pos = -1;
      uint32_t f_len = 0, f_elt = 0, min_len = 0xffffffffu;
      for(uint32_t c0 = 0; c0 < cnt; c0 += 32) {
        const uint32_t p = c0 + lane;
        const bool in = p < cnt;
        const uint32_t slot = cnt - 1 - p;
        int32_t lsr = 0, lpb = 0; uint32_t llen = 0, lelt = 0;
        if(in) { lsr = Lsr[slot]; lpb = Lpb[slot]; llen = Llen[slot]; lelt = Lelt[slot]; }
        bool ok_mer;
        if(win) {
          const int32_t wsr = in ? Lwsr[slot] : kNoWindow;
          ok_mer = wsr == kNoWindow || accept_mer(pb_i, sr_i, Lwpb[slot], wsr, a, b, C);
        } else ok_mer = accept_mer(pb_i, sr_i, lpb, lsr, a, b, C);
        const bool feas = in && sr_i > lsr && ok_mer;
        const unsigned ball = __ballot_sync(MR_FULL_MASK, feas);
        const unsigned limit = ball ? (unsigned)(__ffs(ball) - 1) : 32u;
        // len can exceed 27 bits only for groups of > 2^27 hits, which the batch limits exclude
        const unsigned packed = (in && lane < limit) ? ((llen << 5) | lane) : 0xffffffffu;
        const unsigned bp = __reduce_min_sync(MR_FULL_MASK, packed);
        if(bp != 0xffffffffu && (bp >> 5) < min_len) { min_len = bp >> 5; prev_pos = (int)(c0 + (bp & 31)); }
        if(ball) {
          found = (int)(c0 + limit);
          f_len = __shfl_sync(MR_FULL_MASK, llen, limit);
          f_elt = __shfl_sync(MR_FULL_MASK, lelt, limit);
          break;
        }
      }
      const uint32_t e_len = found >= 0 ? f_len + 1 : 1;
      const uint32_t cs = found >= 0 ? cstart[f_elt] : i;
      if(lane == 0) { pprev[i] = found >= 0 ? f_elt : kNone; cstart[i] = cs; }
      const uint32_t q = (uint32_t)(prev_pos + 1);
      for(uint32_t top = cnt; top > cnt - q; ) {
        const uint32_t lo = (top - (cnt - q)) > 32 ? top - 32 : cnt - q;
        const uint32_t s = lo + lane;
        const bool has = s < top;
        int32_t v0 = 0, v1 = 0, v4 = 0, v5 = 0; uint32_t v2 = 0, v3 = 0;
        if(has) { v0 = Lpb[s]; v1 = Lsr[s]; v2 = Llen[s]; v3 = Lelt[s]; if(win) { v4 = Lwpb[s]; v5 = Lwsr[s]; } }
        __syncwarp();
        if(has) { Lpb[s + 1] = v0; Lsr[s + 1] = v1; Llen[s + 1] = v2; Lelt[s + 1] = v3; if(win) { Lwpb[s + 1] = v4; Lwsr[s + 1] = v5; } }
        __syncwarp();
        top = lo;
      }
      if(lane == 0) {
        const uint32_t s = cnt - q;
        Lpb[s] = pb_i; Lsr[s] = sr_i; Llen[s] = e_len; Lelt[s] = i;
        if(win) {
          // what a hit extending this element will be tested against: the element window - 1 links back, once
          // the chain is long enough for its window to fill
          int32_t wpb = 0, wsr = kNoWindow;
          if(e_len >= window) {
            uint32_t w = i;
            for(uint32_t t = 1; t < window; ++t) w = pprev[w];
            const uint64_t pw = pay[w];
            wpb = (int32_t)(uint32_t)pw; wsr = (int32_t)(uint32_t)(pw >> 32);
          }
          Lwpb[s] = wpb; Lwsr[s] = wsr;
        }
      }
      ++cnt;
      __syncwarp();
      if(longest < e_len) {
        const uint64_t pc = pay[cs];
        if(accept_sequence(pb_i - (int32_t)(uint32_t)pc, sr_i - (int32_t)(uint32_t)(pc >> 32), a)) { longest = e_len; best = i; }
      }
    }
  }
  longest_out = longest;
  best_out = best;
}

// ---------------------------------------------------------------------------------------------
// coords of one group from its chain (chain[t] = group-local hit index, in chain order)
// ---------------------------------------------------------------------------------------------
struct coords_acc {
  // online least squares (x = super-read offset, y = read offset) + the consecutive/cover counters
  double EX = 0, EY = 0, EXX = 0, EXY = 0, VX = 0, CXY = 0, NB = 0;
  uint32_t pb_cons = 0, sr_cons = 0, pb_cover, sr_cover;
  int32_t first_pb = 0, first_sr = 0, ppb = 0, psr = 0;
  long n = 0;
  __device__ __forceinline__ explicit coords_acc(uint32_t k) : pb_cover(k), sr_cover(k) { }
  __device__ __forceinline__ void add(int32_t pb, int32_t so, uint32_t k, double rcp_next) {
    if(n == 0) { first_pb = pb; first_sr = so; }
    else {
      const uint32_t pb_diff = (uint32_t)(pb - ppb), sr_diff = (uint32_t)(so - psr);
      pb_cons += pb_diff == 1; pb_cover += min(k, pb_diff);
      sr_cons += sr_diff == 1; sr_cover += min(k, sr_diff);
    }
    ppb = pb; psr = so;
    const double x = (double)so, y = (double)pb;
    ++n;
    const double dn = (double)n;                       // rcp_next == RN(1 / n)
    const double dX = x - EX;  EX += div_by_count(dX, dn, rcp_next);  const double ndX = x - EX;  VX += dX * ndX;
    const double dY = y - EY;  EY += div_by_count(dY, dn, rcp_next);  const double ndY = y - EY;
    const double dXX = x * x - EXX;  EXX += div_by_count(dXX, dn, rcp_next);
    const double dXY = x * y - EXY;  EXY += div_by_count(dXY, dn, rcp_next);
    CXY += dX * ndY;
    const double t1 = dXY * ndX, t2 = dXX * ndY;
    NB += t1 - t2;
  }
};

// (read, super-read) of a group: the key of its first hit, or -- when groups are rows given by the
// caller (fine pass: a group may be empty) -- the caller's per-group arrays
__device__ __forceinline__ void group_identity(const chain_args& A, uint64_t g, uint64_t gs, uint32_t& read, uint32_t& sr) {
  if(A.group_read) { read = A.group_read[g]; sr = A.group_sr[g]; return; }
  const uint64_t key = A.keys[gs];
  read = (uint32_t)(key >> 32); sr = (uint32_t)key;
}

// canonicalize + filters + survivor append; call from ONE thread per group
__device__ __forceinline__ bool publish_coords(const chain_args& A, uint64_t gs, uint32_t read, uint32_t sr, bool fwd_align,
                                               uint32_t nb, const coords_acc& c, double stretch, double offset, double avg_err,
                                               uint32_t iter = 0) {
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const uint32_t ql = A.sr_len[sr];
  const uint32_t rl = (uint32_t)(A.read_start[read + 1] - A.read_start[read]);
  int32_t rs = c.first_pb, re = c.ppb + (int32_t)k - 1, qs = c.first_sr, qe = c.psr;
  bool rn = false;
  if(qs < 0) {
    if(A.forward) {
      qs = (int32_t)((int64_t)ql + qs - (int64_t)k + 2);
      qe = (int32_t)((int64_t)ql + qe + 1);
      rn = true;
      const double t = stretch * (double)((uint64_t)ql + 1);
      offset -= t - (double)k;
    } else {
      qs = -qs + (int32_t)k - 1;
      qe = -qe;
      stretch = -stretch;
      offset += (double)(k - 1);
    }
  } else {
    qe += (int32_t)k - 1;
  }
  // filters of align_sequence_max (coarse_aligner.cc:51-54); the fine pass keeps every row (fine_aligner.cc:47-49)
  if(!A.no_filter && fabs(stretch) == 0.0) return false;
  if(!A.no_filter) {
    const double drl = (double)rl;
    const double is = fmax(1.0, fmin(drl, stretch + offset));
    const double tq = stretch * (double)ql;
    const double ie = fmax(1.0, fmin(drl, tq + offset));
    const int imp_len = (int)llabs(llrint(ie - is)) + 1;
    if(A.matching_mers != 0.0 && !(A.matching_mers * (double)(uint32_t)((uint32_t)imp_len - k + 1) <= (double)(int)nb)) return false;
    if(A.matching_bases > 0.0 && !(A.matching_bases * (double)(imp_len - 2 * (int)k) <= (double)c.pb_cover)) return false;
  }
  const bool use_bwd = A.forward && !fwd_align;
  uint32_t ilen = 0;
  if(A.unitigs_k && A.unitig_off) {
    const uint64_t u0 = A.unitig_off[sr], u1 = A.unitig_off[sr + 1];
    if(u1 > u0) {
      const uint32_t first_id = (use_bwd ? A.unitig_ids[u1 - 1] : A.unitig_ids[u0]) >> 1;
      if(first_id < A.n_unitigs) ilen = 2 * (uint32_t)(u1 - u0) - 1;
    }
  }
  const survivors& sv = A.sv;
  const unsigned long long slot = atomicAdd(sv.count, 1ULL);
  if(slot < sv.cap) {
    sv.rs[slot] = rs; sv.re[slot] = re; sv.qs[slot] = qs; sv.qe[slot] = qe; sv.nb_mers[slot] = (int32_t)nb;
    sv.pb_cons[slot] = c.pb_cons; sv.sr_cons[slot] = c.sr_cons; sv.pb_cover[slot] = c.pb_cover; sv.sr_cover[slot] = c.sr_cover;
    sv.ql[slot] = ql; sv.sr[slot] = sr; sv.read[slot] = read; sv.info_len[slot] = ilen;
    sv.rn[slot] = rn; sv.use_bwd[slot] = use_bwd;
    sv.stretch[slot] = stretch; sv.offset[slot] = offset; sv.avg_err[slot] = avg_err;
    sv.chain_pos[slot] = gs;
    sv.iter[slot] = iter;
    atomicAdd(sv.info_total, (unsigned long long)ilen);
    atomicAdd(sv.read_cnt + read, 1u);
  }
  return true;
}

// long chains: one warp per group, the lanes fetch 32 hits (and 32 reciprocals) at a time and every
// lane runs the same sequential recurrence on the broadcast values
// WANT_RESULT: broadcast "the row passed the filters" to the whole warp (needed by --max-match only).
// Without it the function ends with lane 0's publish and no warp collective: a version that always
// ended in a __shfl_sync whose result the caller ignored hung on sm_100a (long chains, CUDA 12.9).
template<bool WANT_RESULT>
__device__ __forceinline__ bool finish_group_warp(const chain_args& A, uint64_t gs, uint32_t read, uint32_t sr, bool fwd_align,
                                                  uint32_t nb, uint32_t iter = 0) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const uint64_t* cp = A.chain_pay + gs;          // the chain's (pb, sr) pairs, in chain order
  coords_acc c(k);
  for(uint32_t t0 = 0; t0 < nb; t0 += 32) {
    const uint32_t tl = t0 + lane;
    uint64_t pl = 0;
    if(tl < nb) pl = cp[tl];
    const double rl = 1.0 / (double)(tl + 1);
    const uint32_t m = min(32u, nb - t0);
    for(uint32_t u = 0; u < m; ++u) {
      const uint64_t p = __shfl_sync(MR_FULL_MASK, pl, u);
      c.add((int32_t)(uint32_t)p, (int32_t)(uint32_t)(p >> 32), k, __shfl_sync(MR_FULL_MASK, rl, u));
    }
  }
  double stretch, offset, avg_err;
  if(c.n == 1) { stretch = 1.0; offset = c.EY - c.EX; avg_err = 0; }
  else {
    stretch = c.CXY / c.VX; offset = c.NB / c.VX;
    double e = 0;
    for(uint32_t t0 = 0; t0 < nb; t0 += 32) {
      const uint32_t tl = t0 + lane;
      uint64_t pl = 0;
      if(tl < nb) pl = cp[tl];
      const uint32_t m = min(32u, nb - t0);
      for(uint32_t u = 0; u < m; ++u) {
        const uint64_t p = __shfl_sync(MR_FULL_MASK, pl, u);
        const double x = (double)(int32_t)(uint32_t)(p >> 32), y = (double)(int32_t)(uint32_t)p;
        const double prod = stretch * x;
        e += fabs(prod + offset - y);
      }
    }
    avg_err = e / (double)c.n;
  }
  if(!WANT_RESULT) {
    if(lane == 0) publish_coords(A, gs, read, sr, fwd_align, nb, c, stretch, offset, avg_err, iter);
    return false;
  }
  int passed = 0;
  if(lane == 0) passed = publish_coords(A, gs, read, sr, fwd_align, nb, c, stretch, offset, avg_err, iter) ? 1 : 0;
  __syncwarp();
  return __shfl_sync(MR_FULL_MASK, passed, 0) != 0;
}

// one THREAD per group: 32 independent recurrences per warp instruction.  The chain's pairs are read
// four at a time, the next four already in flight while the current ones are folded in.
__device__ __forceinline__ void finish_group_thread(const chain_args& A, uint64_t gs, uint32_t read, uint32_t sr, bool fwd_align,
                                                    uint32_t nb, uint32_t iter = 0) {
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const uint64_t* cp = A.chain_pay + gs;
  coords_acc c(k);
  uint64_t q[4];
#pragma unroll
  for(int j = 0; j < 4; ++j) q[j] = (uint32_t)j < nb ? cp[j] : 0;
  for(uint32_t t0 = 0; t0 < nb; t0 += 4) {
    uint64_t nq[4];
#pragma unroll
    for(int j = 0; j < 4; ++j) nq[j] = t0 + 4 + j < nb ? cp[t0 + 4 + j] : 0;
#pragma unroll
    for(int j = 0; j < 4; ++j)
      if(t0 + j < nb) c.add((int32_t)(uint32_t)q[j], (int32_t)(uint32_t)(q[j] >> 32), k, rcp_count(t0 + j + 1));
#pragma unroll
    for(int j = 0; j < 4; ++j) q[j] = nq[j];
  }
  double stretch, offset, avg_err;
  if(c.n == 1) { stretch = 1.0; offset = c.EY - c.EX; avg_err = 0; }
  else {
    stretch = c.CXY / c.VX; offset = c.NB / c.VX;
    double e = 0;
    for(uint32_t t = 0; t < nb; ++t) {
      const uint64_t p = cp[t];
      const double x = (double)(int32_t)(uint32_t)(p >> 32), y = (double)(int32_t)(uint32_t)p;
      const double prod = stretch * x;
      e += fabs(prod + offset - y);
    }
    avg_err = e / (double)c.n;
  }
  publish_coords(A, gs, read, sr, fwd_align, nb, c, stretch, offset, avg_err, iter);
}

// a window of the fine pass without any hit: compute_coords_info returns right after the constructor
// (pb_aligner.cc:25-28).  The reference leaves rs, re, qs, qe uninitialised there; they are 0 here.
__device__ __forceinline__ void publish_empty(const chain_args& A, uint64_t gs, uint32_t read, uint32_t sr, uint32_t iter) {
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const survivors& sv = A.sv;
  const unsigned long long slot = atomicAdd(sv.count, 1ULL);
  if(slot < sv.cap) {
    sv.rs[slot] = 0; sv.re[slot] = 0; sv.qs[slot] = 0; sv.qe[slot] = 0; sv.nb_mers[slot] = 0;
    sv.pb_cons[slot] = 0; sv.sr_cons[slot] = 0; sv.pb_cover[slot] = k; sv.sr_cover[slot] = k;
    sv.ql[slot] = A.sr_len[sr]; sv.sr[slot] = sr; sv.read[slot] = read; sv.info_len[slot] = 0;
    sv.rn[slot] = 0; sv.use_bwd[slot] = 0;
    sv.stretch[slot] = 0; sv.offset[slot] = 0; sv.avg_err[slot] = 0;
    sv.chain_pos[slot] = gs;
    sv.iter[slot] = iter;
    atomicAdd(sv.read_cnt + read, 1u);
  }
}

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
// bins groups by size; list c holds the group ids of class c: class c < kSmemTiers holds the groups
// of at most kTierCap[c] hits (and more than the tier below), the last class everything larger
constexpr int kSmemTiers = 9;
constexpr int kClasses = kSmemTiers + 1;
__constant__ uint32_t kTierCap[kSmemTiers] = { 64, 256, 512, 768, 1024, 1536, 2048, 3072, 4096 };
constexpr uint32_t kTierCapHost[kSmemTiers] = { 64, 256, 512, 768, 1024, 1536, 2048, 3072, 4096 };
constexpr uint32_t kTierWarps[kSmemTiers]   = { 8, 8, 4, 4, 2, 1, 1, 1, 1 };       // warps (= groups in flight) per block
// groups of 2 .. kTinyMax hits (chance matches of a 16- or 17-mer: most groups that are not single
// hits) get one THREAD each, list kClasses; a warp per two-hit group would waste 30 lanes on ~800 instructions
constexpr uint32_t kTinyMax = 8;
// Single-hit groups (most groups: spurious k-mer matches) need no chaining at all: their chain is
// hit 0, which this kernel records directly.
// A group whose key carries the super-read index `stray_sr` holds a read's hits that belong to no super-read (their
// k-mer straddles two of them; the per-read sort of group.cu leaves them as the last group of the read's slice):
// it is not chained and yields no row (group_nb = 0).  keys == nullptr: the groups are not keyed by super-read.
__global__ void __launch_bounds__(256) classify_groups_kernel(const uint64_t* __restrict__ group_start, uint64_t ngroups,
                                                               const uint64_t* __restrict__ keys, uint32_t stray_sr,
                                                               const uint64_t* __restrict__ pays, uint64_t* __restrict__ chain_pay,
                                                               uint32_t* __restrict__ group_nb, uint2* __restrict__ tap_lens,
                                                               bool singles_here, bool all_global,
                                                               uint32_t* __restrict__ lists, uint32_t* __restrict__ counts) {
  // (singles_here is false with parity taps or --max-match on: then every group goes to the strand kernels)
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int cls = -1;
  if(g < ngroups) {
    const uint64_t gs = group_start[g];
    const uint64_t n = group_start[g + 1] - gs;
    cls = kSmemTiers;
#pragma unroll
    for(int c = kSmemTiers - 1; c >= 0; --c) if(n <= kTierCap[c]) cls = c;
    if(n == 0) {                                 // a fine-pass window without hits: no chain, a default row
      cls = -1;
      group_nb[g] = 0x80000000u;
    } else if(keys && (uint32_t)keys[gs] == stray_sr) {
      cls = -1;
      group_nb[g] = 0;
      if(tap_lens) tap_lens[g] = make_uint2(0, 0);
    } else if(n == 1 && singles_here) {
      cls = -1;
      const uint64_t p = pays[gs];
      chain_pay[gs] = p;
      group_nb[g] = 1u | ((int32_t)(uint32_t)(p >> 32) > 0 ? 0x80000000u : 0u);
    } else if(all_global) cls = kSmemTiers;      // --window-size > 1: only the global-memory kernel implements it
    else if(n <= kTinyMax && singles_here) cls = kClasses;
  }
  const unsigned lane = threadIdx.x & 31;
#pragma unroll
  for(int c = 0; c <= kClasses; ++c) {
    const unsigned m = __ballot_sync(MR_FULL_MASK, cls == c);
    if(!m) continue;
    unsigned base = 0;
    if(lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(counts + c, __popc(m));
    base = __shfl_sync(MR_FULL_MASK, base, __ffs(m) - 1);
    if(cls == c) lists[(uint64_t)c * ngroups + base + __popc(m & lanemask_lt())] = (uint32_t)g;
  }
}

// chains of the tiny groups: one thread per group runs compute_L_P as written (lis_align.hpp:139-182)
// on arrays of kTinyMax entries
__global__ void __launch_bounds__(128) chain_tiny_kernel(chain_args A, const uint32_t* __restrict__ list,
                                                          const uint32_t* __restrict__ list_count) {
  const uint32_t total = *list_count;
  for(uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < total; w += gridDim.x * blockDim.x) {
    const uint32_t g = list[w];
    const uint64_t gs = A.group_start[g];
    const uint32_t N = (uint32_t)(A.group_start[g + 1] - gs);
    int32_t pb[kTinyMax], sr[kTinyMax];
    uint8_t len[kTinyMax], cstart[kTinyMax], pprev[kTinyMax], L[kTinyMax];
    for(uint32_t i = 0; i < N; ++i) { const uint64_t p = A.pays[gs + i]; pb[i] = (int32_t)(uint32_t)p; sr[i] = (int32_t)(uint32_t)(p >> 32); }
    uint32_t longest[2] = { 0, 0 }, best[2] = { 0, 0 };
    for(int s = 0; s < 2; ++s) {
      uint32_t cnt = 0;
      for(uint32_t i = 0; i < N; ++i) {
        if((sr[i] < 0) != (s == 1)) continue;
        int found = -1, prev = -1;
        uint32_t min_len = 0xffffffffu;
        for(uint32_t p = 0; p < cnt; ++p) {                 // list order, front first
          const uint32_t j = L[p];
          if(sr[i] > sr[j] && accept_mer(pb[i], sr[i], pb[j], sr[j], A.a, A.b, A.C)) { found = (int)p; break; }
          if(len[j] < min_len) { min_len = len[j]; prev = (int)p; }
        }
        const uint32_t fj = found >= 0 ? L[found] : 0;
        const uint32_t e_len = found >= 0 ? len[fj] + 1u : 1u;
        const uint32_t cs = found >= 0 ? cstart[fj] : i;
        len[i] = (uint8_t)e_len; cstart[i] = (uint8_t)cs; pprev[i] = found >= 0 ? (uint8_t)fj : (uint8_t)0xff;
        for(int p = (int)cnt; p > prev + 1; --p) L[p] = L[p - 1];
        L[prev + 1] = (uint8_t)i;
        ++cnt;
        if(longest[s] < e_len && accept_sequence(pb[i] - pb[cs], sr[i] - sr[cs], A.a)) { longest[s] = e_len; best[s] = i; }
      }
    }
    const bool fwd_align = longest[0] >= longest[1];
    const uint32_t nb = fwd_align ? longest[0] : longest[1];
    uint32_t cur = fwd_align ? best[0] : best[1];
    for(uint32_t t = 0; t < nb; ++t) {
      A.chain_pay[gs + nb - 1 - t] = (uint64_t)(uint32_t)pb[cur] | ((uint64_t)(uint32_t)sr[cur] << 32);
      cur = pprev[cur];
    }
    A.group_nb[g] = nb | (fwd_align ? 0x80000000u : 0u);
  }
}

// strands of the groups of one size class, out of shared memory: one warp per group, `cap` hits of
// room per warp
template<bool TAPS>
__global__ void __launch_bounds__(256) chain_coords_smem_kernel(chain_args A, const uint32_t* __restrict__ list,
                                                                const uint32_t* __restrict__ list_count,
                                                                uint32_t* __restrict__ cursor, uint32_t cap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  unsigned char* mine_raw = smem_raw + warp_store_bytes(cap, TAPS) * wib;
  const warp_store S(mine_raw, cap);
  uint16_t* sub = TAPS ? reinterpret_cast<uint16_t*>(mine_raw + warp_store_bytes(cap, false)) : nullptr;
  const uint32_t total = *list_count;
  while(true) {
    uint32_t w = 0;
    if(lane == 0) w = atomicAdd(cursor, 1u);              // dynamic work distribution, one group per grab
    w = __shfl_sync(MR_FULL_MASK, w, 0);
    if(w >= total) break;
    const uint32_t g = list[w];
    const uint64_t gs = A.group_start[g];
    const uint32_t N = (uint32_t)(A.group_start[g + 1] - gs);
    const long long dbg_t0 = A.dbg_cycles ? clock64() : 0;
    uint32_t len_f = 0, best_f = 0, len_b = 0, best_b = 0;
    chain_strand_smem<TAPS>(A.pays + gs, N, false, S, sub, A.a, A.b, A.C, len_f, best_f);
    __syncwarp();
    chain_strand_smem<TAPS>(A.pays + gs, N, true, S, sub, A.a, A.b, A.C, len_b, best_b);
    __syncwarp();
    const bool fwd_align = len_f >= len_b;
    const uint32_t nb = fwd_align ? len_f : len_b;
    if(TAPS) {
      if(lane == 0) {
        A.tap_lens[g] = make_uint2(len_f, len_b);
        uint32_t cur = best_f;
        for(uint32_t t = 0; t < len_f; ++t) { A.tap_cf[gs + len_f - 1 - t] = sub[cur]; cur = S.pprev[cur]; }
        cur = best_b;
        for(uint32_t t = 0; t < len_b; ++t) { A.tap_cb[gs + len_b - 1 - t] = sub[cur]; cur = S.pprev[cur]; }
      }
      __syncwarp();
    }
    // L is dead: its pb[] array becomes the chain, in order
    uint32_t* chain = reinterpret_cast<uint32_t*>(S.pb);
    if(lane == 0) {
      uint32_t cur = fwd_align ? best_f : best_b;
      for(uint32_t t = 0; t < nb; ++t) { chain[nb - 1 - t] = cur; cur = S.pprev[cur]; }
    }
    __syncwarp();
    // publish the chain's (pb, sr) pairs in chain order and the group's verdict; the coords are
    // computed by finish_*_kernel at full occupancy
    for(uint32_t t = lane; t < nb; t += 32) A.chain_pay[gs + t] = A.pays[gs + chain[t]];
    if(lane == 0) {
      A.group_nb[g] = nb | (fwd_align ? 0x80000000u : 0u);
      if(A.dbg_cycles) A.dbg_cycles[g] = (uint32_t)(clock64() - dbg_t0);
      if(nb > kThreadFinishLongMax) A.long_list[atomicAdd(A.long_count, 1u)] = g;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) chain_coords_global_kernel(chain_args A, const uint32_t* __restrict__ list,
                                                                   const uint32_t* __restrict__ list_count,
                                                                   uint32_t* __restrict__ cursor) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t total = list ? *list_count : (uint32_t)A.ngroups;
  while(true) {
    uint32_t w = 0;
    if(lane == 0) w = atomicAdd(cursor, 1u);
    w = __shfl_sync(MR_FULL_MASK, w, 0);
    if(w >= total) break;
    const uint32_t g = list ? list[w] : w;
    const uint64_t gs = A.group_start[g];
    const uint32_t N = (uint32_t)(A.group_start[g + 1] - gs);
    uint32_t len_f = 0, best_f = 0, len_b = 0, best_b = 0;
    chain_strand_global(A.pays + gs, N, false, A.cb, gs, A.a, A.b, A.C, len_f, best_f, A.tap_sub, nullptr, A.window);
    __syncwarp();
    chain_strand_global(A.pays + gs, N, true, A.cb, gs, A.a, A.b, A.C, len_b, best_b, A.tap_sub, nullptr, A.window);
    __syncwarp();
    const bool fwd_align = len_f >= len_b;
    const uint32_t nb = fwd_align ? len_f : len_b;
    uint32_t* chain = A.cb.Lelt + gs;          // L is dead now: reuse as the chain, in order
    uint32_t* pprev = A.cb.pprev + gs;
    if(A.tap_lens) {
      if(lane == 0) {
        A.tap_lens[g] = make_uint2(len_f, len_b);
        uint32_t cur = best_f;
        for(uint32_t t = 0; t < len_f; ++t) { A.tap_cf[gs + len_f - 1 - t] = A.tap_sub[gs + cur]; cur = pprev[cur]; }
        cur = best_b;
        for(uint32_t t = 0; t < len_b; ++t) { A.tap_cb[gs + len_b - 1 - t] = A.tap_sub[gs + cur]; cur = pprev[cur]; }
      }
      __syncwarp();
    }
    if(lane == 0) {
      uint32_t cur = fwd_align ? best_f : best_b;
      for(uint32_t t = 0; t < nb; ++t) { chain[nb - 1 - t] = cur; cur = pprev[cur]; }
    }
    __syncwarp();
    for(uint32_t t = lane; t < nb; t += 32) A.chain_pay[gs + t] = A.pays[gs + chain[t]];
    if(lane == 0) {
      A.group_nb[g] = nb | (fwd_align ? 0x80000000u : 0u);
      if(nb > kThreadFinishLongMax) A.long_list[atomicAdd(A.long_count, 1u)] = g;
    }
    __syncwarp();
  }
}

// coords, one thread per group: warps hold 32 chains, the FP64 recurrence of each is latency bound
// and 32 of them share every instruction.
// (1) every group of at most max_group hits, in group order (neighbouring threads read neighbouring chains)
__global__ void __launch_bounds__(128) finish_small_groups_kernel(chain_args A, uint32_t max_group) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(g >= A.ngroups) return;
  const uint64_t gs = A.group_start[g];
  if(A.group_start[g + 1] - gs > max_group) return;
  const uint32_t v = A.group_nb[g];
  if(v == 0) return;                             // hits that belong to no super-read (classify_groups_kernel)
  uint32_t read, sr;
  group_identity(A, g, gs, read, sr);
  const uint32_t iter = A.group_iter ? A.group_iter[g] : 0;
  if((v & 0x7fffffffu) == 0) { publish_empty(A, gs, read, sr, iter); return; }
  finish_group_thread(A, gs, read, sr, (v >> 31) != 0, v & 0x7fffffffu, iter);
}
// (2) the groups of one size class, right behind the kernel that chained them (chains longer than
// hi went to the long list).  A warp takes 32 chains, one per lane; each chain is a private stream
// of 8-byte pairs, so the lanes do not read them themselves (32 different cache lines per load, and
// next to the chaining kernels the L1 is a few KB): the warp copies 16 pairs of every chain into a
// shared-memory tile with coalesced cp.async, the next tile in flight while the current one is folded in.
constexpr int kTileE = 16;
// Groups of at most `lo` hits are left to finish_small_groups_kernel (they only appear in a class list here when
// --window-size > 1 sends every group through the global-memory chaining kernel).
__global__ void __launch_bounds__(128) finish_tile_kernel(chain_args A, const uint32_t* __restrict__ list,
                                                           const uint32_t* __restrict__ list_count, uint32_t hi, uint32_t lo) {
  __shared__ uint64_t tile[4][2][32][kTileE + 1];      // + 1: lane j reads row j, 17 x 8 B apart -> no bank conflicts
  const unsigned lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t total = *list_count;
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const uint32_t stride = gridDim.x * 4 * 32;
  for(uint32_t i0 = (blockIdx.x * 4 + wib) * 32; i0 < total; i0 += stride) {
    const uint32_t i = i0 + lane;
    uint32_t v = 0, nb = 0, g = 0;
    uint64_t gs = 0;
    if(i < total) {
      g = list[i];
      v = A.group_nb[g]; nb = v & 0x7fffffffu;
      if(nb > hi) nb = 0;
      gs = A.group_start[g];
      if(A.group_start[g + 1] - gs <= lo) nb = 0;
    }
    const uint32_t maxnb = __reduce_max_sync(MR_FULL_MASK, nb);
    if(maxnb == 0) continue;
    auto issue = [&](uint32_t t0, int buf) {
#pragma unroll 4
      for(int it = 0; it < 16; ++it) {                  // two chains per step, 16 lanes (128 B) each
        const int jj = it * 2 + (int)(lane >> 4);
        const uint64_t bj = __shfl_sync(MR_FULL_MASK, gs, jj);
        const uint32_t nj = __shfl_sync(MR_FULL_MASK, nb, jj);
        const uint32_t e = t0 + (lane & 15);
        if(e < nj) cp_async8(&tile[wib][buf][jj][lane & 15], A.chain_pay + bj + e);
      }
      cp_async_commit();
    };
    coords_acc c(k);
    int buf = 0;
    issue(0, 0);
    for(uint32_t t0 = 0; t0 < maxnb; t0 += kTileE) {
      if(t0 + kTileE < maxnb) { issue(t0 + kTileE, buf ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      __syncwarp();
#pragma unroll 4
      for(uint32_t e = 0; e < kTileE; ++e) {
        if(t0 + e < nb) {
          const uint64_t p = tile[wib][buf][lane][e];
          c.add((int32_t)(uint32_t)p, (int32_t)(uint32_t)(p >> 32), k, rcp_count(t0 + e + 1));
        }
      }
      __syncwarp();
      buf ^= 1;
    }
    double stretch = 1.0, offset = c.EY - c.EX, avg_err = 0;
    const bool fit = nb > 1;
    if(fit) { stretch = c.CXY / c.VX; offset = c.NB / c.VX; }
    if(__any_sync(MR_FULL_MASK, fit)) {
      double err = 0;
      buf = 0;
      issue(0, 0);
      for(uint32_t t0 = 0; t0 < maxnb; t0 += kTileE) {
        if(t0 + kTileE < maxnb) { issue(t0 + kTileE, buf ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
        __syncwarp();
#pragma unroll 4
        for(uint32_t e = 0; e < kTileE; ++e) {
          if(t0 + e < nb) {
            const uint64_t p = tile[wib][buf][lane][e];
            const double x = (double)(int32_t)(uint32_t)(p >> 32), y = (double)(int32_t)(uint32_t)p;
            const double prod = stretch * x;
            err += fabs(prod + offset - y);
          }
        }
        __syncwarp();
        buf ^= 1;
      }
      if(fit) avg_err = err / (double)c.n;
    }
    if(nb != 0) {
      uint32_t read, sr;
      group_identity(A, g, gs, read, sr);
      publish_coords(A, gs, read, sr, (v >> 31) != 0, nb, c, stretch, offset, avg_err, A.group_iter ? A.group_iter[g] : 0);
    }
  }
}

// The same job with FOUR lanes per chain, one for each of the running means the online least squares keeps (EX, EY,
// EXX, EXY: four independent recurrences, each five dependent FP64 operations per hit): 21 FP64 instructions per hit
// on the critical path instead of 41, eight chains per warp, no shared memory.  An experiment kept behind
// MR_FINISH_QUAD=1: it shortens a lone chain but costs twice the FP64 issue slots per chain, and the phase as a whole
// is bound by those (see launch_chain).  Lane 0 of a quad also owns VX and the super-read counters, lane 1 CXY
// and the read counters, lane 3 NB; the products that mix two recurrences (dX ndY, dXY ndX, dXX ndY) travel by
// shuffle.  Every quantity sees exactly the operations, in the order, of coords_acc::add.
__global__ void __launch_bounds__(128) finish_quad_kernel(chain_args A, const uint32_t* __restrict__ list,
                                                           const uint32_t* __restrict__ list_count, uint32_t hi, uint32_t lo) {
  const unsigned lane = threadIdx.x & 31, q = lane & 3, qbase = lane & ~3u;
  const uint32_t total = *list_count;
  const uint32_t k = A.align_k ? A.align_k : A.iv.k;
  const uint32_t stride = gridDim.x * 4 * 8;
  for(uint32_t i0 = (blockIdx.x * 4 + (threadIdx.x >> 5)) * 8; i0 < total; i0 += stride) {
    const uint32_t i = i0 + (lane >> 2);
    uint32_t v = 0, nb = 0, g = 0;
    uint64_t gs = 0;
    if(i < total) {
      g = list[i];
      v = A.group_nb[g]; nb = v & 0x7fffffffu;
      if(nb > hi) nb = 0;
      gs = A.group_start[g];
      if(A.group_start[g + 1] - gs <= lo) nb = 0;
    }
    const uint32_t maxnb = __reduce_max_sync(MR_FULL_MASK, nb);
    if(maxnb == 0) continue;
    const uint64_t* cp = A.chain_pay + gs;
    double E = 0, acc = 0;
    uint32_t cons = 0, cover = k;
    int32_t prevw = 0;
    uint64_t nxt[8];
#pragma unroll
    for(int e = 0; e < 8; ++e) nxt[e] = (uint32_t)e < nb ? cp[e] : 0;
    for(uint32_t t0 = 0; t0 < maxnb; t0 += 8) {
      uint64_t cur[8];
#pragma unroll
      for(int e = 0; e < 8; ++e) { cur[e] = nxt[e]; nxt[e] = t0 + 8 + e < nb ? cp[t0 + 8 + e] : 0; }
#pragma unroll
      for(int e = 0; e < 8; ++e) {
        const uint32_t t = t0 + e;
        const bool act = t < nb;
        const int32_t pb = (int32_t)(uint32_t)cur[e], so = (int32_t)(uint32_t)(cur[e] >> 32);
        const double x = (double)so, y = (double)pb;
        const double xx = x * x, xy = x * y;
        const double val = q == 0 ? x : (q == 1 ? y : (q == 2 ? xx : xy));
        const double dn = (double)(t + 1), r = rcp_count(t + 1);
        const double d = val - E;
        const double En = E + div_by_count(d, dn, r);
        const double nd = val - En;
        const double dX = __shfl_sync(MR_FULL_MASK, d, qbase);                          // lane 1 needs dX
        const double ndo = __shfl_sync(MR_FULL_MASK, nd, qbase + (q == 2 ? 1u : 0u));     // lane 2: ndY, lane 3: ndX
        const double a = q == 1 ? dX : d, b = q >= 2 ? ndo : nd;
        const double prod = a * b;                       // lane 0: dX ndX, lane 1: dX ndY, lane 2: dXX ndY, lane 3: dXY ndX
        const double t2 = __shfl_sync(MR_FULL_MASK, prod, qbase + 2);
        const double add = q == 3 ? prod - t2 : prod;
        const int32_t w = q == 1 ? pb : so;
        if(act) {
          E = En;
          acc += add;
          if(t != 0) {
            const uint32_t diff = (uint32_t)(w - prevw);
            cons += diff == 1; cover += min(k, diff);
          }
          prevw = w;
        }
      }
    }
    const double VX = __shfl_sync(MR_FULL_MASK, acc, qbase), CXY = __shfl_sync(MR_FULL_MASK, acc, qbase + 1), NB = __shfl_sync(MR_FULL_MASK, acc, qbase + 3);
    const double EX = __shfl_sync(MR_FULL_MASK, E, qbase), EY = __shfl_sync(MR_FULL_MASK, E, qbase + 1);
    double stretch = 1.0, offset = EY - EX, avg_err = 0;
    const bool fit = nb > 1;
    if(fit) { stretch = CXY / VX; offset = NB / VX; }
    if(__any_sync(MR_FULL_MASK, fit)) {                  // every lane of the quad runs the same sum
      double err = 0;
#pragma unroll
      for(int e = 0; e < 8; ++e) nxt[e] = (uint32_t)e < nb ? cp[e] : 0;
      for(uint32_t t0 = 0; t0 < maxnb; t0 += 8) {
        uint64_t cur[8];
#pragma unroll
        for(int e = 0; e < 8; ++e) { cur[e] = nxt[e]; nxt[e] = t0 + 8 + e < nb ? cp[t0 + 8 + e] : 0; }
#pragma unroll
        for(int e = 0; e < 8; ++e) {
          if(t0 + e < nb) {
            const double x = (double)(int32_t)(uint32_t)(cur[e] >> 32), y = (double)(int32_t)(uint32_t)cur[e];
            const double prod = stretch * x;
            err += fabs(prod + offset - y);
          }
        }
      }
      if(fit) avg_err = err / (double)(long)nb;
    }
    const uint32_t pb_cons = __shfl_sync(MR_FULL_MASK, cons, qbase + 1), pb_cover = __shfl_sync(MR_FULL_MASK, cover, qbase + 1);
    if(nb != 0 && q == 0) {
      coords_acc c(k);
      const uint64_t p0 = cp[0], p1 = cp[nb - 1];
      c.first_pb = (int32_t)(uint32_t)p0; c.first_sr = (int32_t)(uint32_t)(p0 >> 32);
      c.ppb = (int32_t)(uint32_t)p1; c.psr = (int32_t)(uint32_t)(p1 >> 32);
      c.pb_cons = pb_cons; c.pb_cover = pb_cover; c.sr_cons = cons; c.sr_cover = cover;
      c.n = (long)nb;
      uint32_t read, sr;
      group_identity(A, g, gs, read, sr);
      publish_coords(A, gs, read, sr, (v >> 31) != 0, nb, c, stretch, offset, avg_err, A.group_iter ? A.group_iter[g] : 0);
    }
  }
}

// ... and of the very long chains: one warp per group
__global__ void __launch_bounds__(128) finish_warp_kernel(chain_args A) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t total = *A.long_count;
  while(true) {
    uint32_t w = 0;
    if(lane == 0) w = atomicAdd(A.long_cursor, 1u);
    w = __shfl_sync(MR_FULL_MASK, w, 0);
    if(w >= total) break;
    const uint32_t g = A.long_list[w];
    const uint32_t v = A.group_nb[g];
    const uint64_t gs = A.group_start[g];
    uint32_t read, sr;
    group_identity(A, g, gs, read, sr);
    finish_group_warp<false>(A, gs, read, sr, (v >> 31) != 0, v & 0x7fffffffu, A.group_iter ? A.group_iter[g] : 0);
  }
}

// --max-match (coarse_aligner.cc:56-57, pb_aligner.hpp:47-92): after a row passes the filters the
// chain of the strictly-longer-forward-else-backward list is removed from its list, that list is
// chained again and the group is evaluated again, until a row fails.  One warp per group out of
// global scratch; successive chains of a group are stored back to back in its chain_pay slice.
// TAPS (parity taps on): record the state the loop ends in, as the reference's --details prints it: each strand's
// latest chain, numbered within that strand's hits not yet removed.  A strand loses hits only right before it is
// chained again, so its latest numbering is the one of its final hit list.  (A kernel of its own: the taps' extra live
// values would make the production kernel spill more.)
template<bool TAPS>
__global__ void __launch_bounds__(128) chain_maxmatch_kernel(chain_args A, uint8_t* __restrict__ removed, uint32_t* __restrict__ cursor) {
  const unsigned lane = threadIdx.x & 31;
  while(true) {
    uint32_t g = 0;
    if(lane == 0) g = atomicAdd(cursor, 1u);
    g = __shfl_sync(MR_FULL_MASK, g, 0);
    if(g >= A.ngroups) break;
    const uint64_t gs = A.group_start[g];
    const uint32_t N = (uint32_t)(A.group_start[g + 1] - gs);
    const uint64_t key = A.keys[gs];
    const uint32_t read = (uint32_t)(key >> 32), sr = (uint32_t)key;
    if(sr == A.iv.nseq_all) continue;              // hits that belong to no super-read
    uint8_t* rem = removed + gs;
    for(uint32_t t = lane; t < N; t += 32) rem[t] = 0;
    __syncwarp();
    uint32_t len_f = 0, best_f = 0, len_b = 0, best_b = 0, used = 0;
    chain_strand_global(A.pays + gs, N, false, A.cb, gs, A.a, A.b, A.C, len_f, best_f, TAPS ? A.tap_sub : nullptr, rem, A.window);
    __syncwarp();
    chain_strand_global(A.pays + gs, N, true, A.cb, gs, A.a, A.b, A.C, len_b, best_b, TAPS ? A.tap_sub : nullptr, rem, A.window);
    __syncwarp();
    uint32_t* pprev = A.cb.pprev + gs;
    uint32_t* chain = A.cb.Lelt + gs;            // L is dead between chainings
    for(uint32_t iter = 0; ; ++iter) {
      const bool fwd_align = len_f >= len_b;
      const uint32_t nb = fwd_align ? len_f : len_b;
      if(nb == 0) break;
      if(lane == 0) {
        uint32_t cur = fwd_align ? best_f : best_b;
        for(uint32_t t = 0; t < nb; ++t) { chain[nb - 1 - t] = cur; cur = pprev[cur]; }
      }
      __syncwarp();
      for(uint32_t t = lane; t < nb; t += 32) A.chain_pay[gs + used + t] = A.pays[gs + chain[t]];
      __syncwarp();
      if(!finish_group_warp<true>(A, gs + used, read, sr, fwd_align, nb, iter)) break;
      used += nb;
      // discard_update_LIS: the forward list only if it is STRICTLY longer, else the backward one
      const bool drop_fwd = len_f > len_b;
      const uint32_t dn = drop_fwd ? len_f : len_b;
      if(lane == 0) {
        uint32_t cur = drop_fwd ? best_f : best_b;
        for(uint32_t t = 0; t < dn; ++t) { rem[cur] = 1; cur = pprev[cur]; }
      }
      __syncwarp();
      if(drop_fwd) chain_strand_global(A.pays + gs, N, false, A.cb, gs, A.a, A.b, A.C, len_f, best_f, TAPS ? A.tap_sub : nullptr, rem, A.window);
      else         chain_strand_global(A.pays + gs, N, true, A.cb, gs, A.a, A.b, A.C, len_b, best_b, TAPS ? A.tap_sub : nullptr, rem, A.window);
      __syncwarp();
    }
    if(TAPS) {
      if(lane == 0) {
        A.tap_lens[g] = make_uint2(len_f, len_b);
        uint32_t cur = best_f;
        for(uint32_t t = 0; t < len_f; ++t) { A.tap_cf[gs + len_f - 1 - t] = A.tap_sub[gs + cur]; cur = pprev[cur]; }
        cur = best_b;
        for(uint32_t t = 0; t < len_b; ++t) { A.tap_cb[gs + len_b - 1 - t] = A.tap_sub[gs + cur]; cur = pprev[cur]; }
      }
      __syncwarp();
    }
  }
}

template<bool TAPS>
int launch_smem(mr_context* ctx, cudaStream_t st, const chain_args& A, int tier, const uint32_t* list, const uint32_t* count, uint32_t* cursor) {
  const uint32_t cap = kTierCapHost[tier], warps = kTierWarps[tier];
  const size_t smem = warp_store_bytes(cap, TAPS) * warps;
  MR_CUDA(ctx, cudaFuncSetAttribute(chain_coords_smem_kernel<TAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)warp_store_bytes(4096, TAPS)));
  // as many blocks as one SM can hold at a time (shared memory, 64 warps, 32 blocks), on every SM
  const size_t per_sm = 227 * 1024;
  const uint32_t fit = (uint32_t)std::min<size_t>(std::min<size_t>(per_sm / (smem + 1024), 64 / warps), 32);
  chain_coords_smem_kernel<TAPS><<<ctx->sm_count * std::max(fit, 1u), warps * 32, smem, st>>>(A, list, count, cursor, cap);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

} // namespace

// scratch `lists`: (kClasses + 3) x ngroups uint32 (size classes, tiny groups, long-chain list, verdicts)
// + 32 uint32 counters (class counts 0..9, tiny count 10, class cursors 16..25, long count 28, long
// cursor 29, max-match cursor 30)
// MR_TRACE=1: synchronise after every chain-phase kernel and name it on stderr
static const bool g_chain_trace = getenv("MR_TRACE") != nullptr;
static double trace_now() { timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec + 1e-9 * t.tv_nsec; }
static double g_trace_t0 = 0;
#define CHAIN_TRACE(st, name) do { if(g_chain_trace) { cudaError_t e_ = cudaStreamSynchronize(st); const double n_ = trace_now(); \
  fprintf(stderr, "[mr]   %-34s %8.3f ms  %s\n", name, 1e3 * (n_ - g_trace_t0), cudaGetErrorString(e_)); fflush(stderr); g_trace_t0 = trace_now(); } } while(0)

// MR_TRACE_TIMELINE=1: timing events around every chain-phase kernel, no extra synchronisation; the
// start / end of each kernel relative to the start of the phase is printed once the phase is over
static const bool g_chain_timeline = getenv("MR_TRACE_TIMELINE") != nullptr;
struct timeline_t {
  struct item { std::string name; cudaEvent_t b, e; };
  std::vector<item> items;
  cudaEvent_t origin = nullptr;
  void begin(cudaStream_t st) { if(!g_chain_timeline) return; cudaEventCreate(&origin); cudaEventRecord(origin, st); }
  void open(const char* name, cudaStream_t st) { if(!g_chain_timeline) return; item it; it.name = name; cudaEventCreate(&it.b); cudaEventCreate(&it.e); cudaEventRecord(it.b, st); items.push_back(it); }
  void close(cudaStream_t st) { if(!g_chain_timeline) return; cudaEventRecord(items.back().e, st); }
  void report() {
    if(!g_chain_timeline) return;
    cudaDeviceSynchronize();
    for(auto& it : items) {
      float b = 0, e = 0;
      cudaEventElapsedTime(&b, origin, it.b); cudaEventElapsedTime(&e, origin, it.e);
      fprintf(stderr, "[mr]   timeline %-28s %8.3f -> %8.3f ms\n", it.name.c_str(), b, e);
      cudaEventDestroy(it.b); cudaEventDestroy(it.e);
    }
    cudaEventDestroy(origin); items.clear();
  }
};

int launch_chain(mr_context* ctx, chain_args A, dev_buf& lists) {
  if(A.ngroups == 0) return MR_OK;
  if(A.ngroups >= (1ULL << 32)) return ctx->fail(MR_ELIMIT, "more than 2^32 (read, super-read) groups in one batch");
  const uint64_t G = A.ngroups;
  MR_TRY(lists.ensure(ctx, ((kClasses + 3) * G + 32) * sizeof(uint32_t)));
  uint32_t* cls = lists.as<uint32_t>();
  uint32_t* ctr = cls + (kClasses + 3) * G;
  A.long_list = cls + (kClasses + 1) * G; A.group_nb = cls + (kClasses + 2) * G; A.long_count = ctr + 28; A.long_cursor = ctr + 29;
  MR_CUDA(ctx, cudaMemsetAsync(ctr, 0, 32 * sizeof(uint32_t), ctx->stream));
  if(!ctx->chain_tables) {
    std::vector<double> rcp(kRcpMax + 1, 0.0);
    for(uint32_t n = 1; n <= kRcpMax; ++n) rcp[n] = 1.0 / (double)n;
    MR_CUDA(ctx, cudaMemcpyToSymbol(kRcpTable, rcp.data(), rcp.size() * sizeof(double)));
    ctx->chain_tables = true;
  }
  static dev_buf dbg;
  if(g_chain_trace && getenv("MR_TRACE_CYCLES")) { MR_TRY(dbg.ensure(ctx, G * 4)); cudaMemset(dbg.p, 0, G * 4); A.dbg_cycles = dbg.as<uint32_t>(); }
  if(g_chain_trace) { cudaStreamSynchronize(ctx->stream); g_trace_t0 = trace_now(); }
  // (with parity taps on, single-hit groups also go through the strand kernels so that their taps get written)
  classify_groups_kernel<<<div_up(G, 256), 256, 0, ctx->stream>>>(A.group_start, G, A.group_read ? nullptr : A.keys, A.iv.nseq_all,
                                                                  A.pays, A.chain_pay, A.group_nb, A.tap_lens,
                                                                  A.tap_lens == nullptr && !A.max_match, A.window > 1, cls, ctr);
  MR_LAUNCHED(ctx);
  CHAIN_TRACE(ctx->stream, "classify");
  if(A.max_match) {
    if(A.tap_lens) chain_maxmatch_kernel<true><<<ctx->sm_count * 8, 128, 0, ctx->stream>>>(A, A.removed, ctr + 30);
    else            chain_maxmatch_kernel<false><<<ctx->sm_count * 8, 128, 0, ctx->stream>>>(A, A.removed, ctr + 30);
    MR_LAUNCHED(ctx);
    return MR_OK;
  }
  const bool taps = A.tap_lens != nullptr;
  // Every size class is latency bound (a group is a sequential walk) and limited by the shared
  // memory its tier needs; the tiers run on separate streams, largest groups first, so that together
  // they fill the SMs, and each is followed on its stream by the kernel that turns its chains into coords.
  cudaStream_t s0 = ctx->stream;
  MR_CUDA(ctx, cudaEventRecord(ctx->ev[0], s0));
  char label[64];
  timeline_t tl;
  tl.begin(s0);
  for(int c = kClasses - 1; c >= 0; --c) {
    cudaStream_t st = c == 0 ? s0 : ctx->aux[c - 1];
    if(c != 0) MR_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev[0], 0));
    const uint32_t* list = cls + (uint64_t)c * G;
    if(c == 0 && !taps) {
      tl.open("tiny groups", st);
      chain_tiny_kernel<<<ctx->sm_count * 8, 128, 0, st>>>(A, cls + (uint64_t)kClasses * G, ctr + kClasses);
      MR_LAUNCHED(ctx);
      tl.close(st);
      CHAIN_TRACE(st, "tiny groups");
    }
    snprintf(label, sizeof label, "strands %d", c); tl.open(label, st);
    if(c == kSmemTiers) {
      chain_coords_global_kernel<<<ctx->sm_count * 4, 128, 0, st>>>(A, list, ctr + c, ctr + 16 + c);
      MR_LAUNCHED(ctx);
    } else if(taps) { MR_TRY(launch_smem<true>(ctx, st, A, c, list, ctr + c, ctr + 16 + c)); }
    else            { MR_TRY(launch_smem<false>(ctx, st, A, c, list, ctr + c, ctr + 16 + c)); }
    tl.close(st);
    if(g_chain_trace) { snprintf(label, sizeof label, "strands, tier %d (<= %u hits)", c, c < kSmemTiers ? kTierCapHost[c] : 0u); CHAIN_TRACE(st, label); }
    snprintf(label, sizeof label, "finish %d", c); tl.open(label, st);
    if(c != 0) {
      // MR_FINISH_QUAD=1: four lanes per chain instead of a thread per chain.  Measured on B200 (yeast shape): the
      // longest tier alone 0.40 ms against 0.34, the whole phase 28.4 ms per step against 25.4 -- FP64 issue slots
      // are the scarce resource, and the quad form spends 1.75 FP64 warp instructions per hit and chain where the
      // thread form spends 0.8.
      static const bool tile_finish = !(getenv("MR_FINISH_QUAD") && atoi(getenv("MR_FINISH_QUAD")) != 0);
      // The coords kernel runs on a stream of the highest priority: the chaining kernels of the other tiers are
      // persistent and fill every SM, and their blocks still waiting for a slot would otherwise be served before the
      // coords blocks of a tier that is already chained (timeline: coords of the longest tier ready at 0.16 ms, done
      // at 1.1).  MR_FINISH_PRIORITY=0: the tier's own stream.
      static const bool prio = !(getenv("MR_FINISH_PRIORITY") && atoi(getenv("MR_FINISH_PRIORITY")) == 0);
      cudaStream_t fs = st;
      if(prio && ctx->hi[c - 1]) {
        fs = ctx->hi[c - 1];
        MR_CUDA(ctx, cudaEventRecord(ctx->ev_hi[c - 1], st));
        MR_CUDA(ctx, cudaStreamWaitEvent(fs, ctx->ev_hi[c - 1], 0));
      }
      const uint32_t lo = c == kSmemTiers && A.window > 1 ? kTierCapHost[0] : 0u;
      if(tile_finish) finish_tile_kernel<<<ctx->sm_count * 4, 128, 0, fs>>>(A, list, ctr + c, kThreadFinishLongMax, lo);
      else            finish_quad_kernel<<<ctx->sm_count * 8, 128, 0, fs>>>(A, list, ctr + c, kThreadFinishLongMax, lo);
      MR_LAUNCHED(ctx);
      tl.close(fs);
      if(g_chain_trace) { snprintf(label, sizeof label, "finish, tier %d", c); CHAIN_TRACE(fs, label); }
      MR_CUDA(ctx, cudaEventRecord(ctx->ev[c], fs));
    } else {
      // (--window-size > 1: the small groups were chained by the global-memory kernel on its own stream)
      if(A.window > 1) MR_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev[kSmemTiers], 0));
      finish_small_groups_kernel<<<div_up(G, 128), 128, 0, st>>>(A, kTierCapHost[0]);
      MR_LAUNCHED(ctx);
      tl.close(st);
      CHAIN_TRACE(st, "finish, small groups");
    }
  }
  for(int c = 1; c < kClasses; ++c) MR_CUDA(ctx, cudaStreamWaitEvent(s0, ctx->ev[c], 0));
  tl.open("finish warp", s0);
  finish_warp_kernel<<<ctx->sm_count * 8, 128, 0, s0>>>(A);      // chains too long for one thread
  MR_LAUNCHED(ctx);
  tl.close(s0);
  tl.report();
  CHAIN_TRACE(s0, "finish, warp per chain");
  if(g_chain_trace && A.dbg_cycles) {
    cudaDeviceSynchronize();
    std::vector<uint32_t> cyc(G), nbv(G); std::vector<uint64_t> gs(G + 1);
    cudaMemcpy(cyc.data(), A.dbg_cycles, G * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(nbv.data(), A.group_nb, G * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(gs.data(), A.group_start, (G + 1) * 8, cudaMemcpyDeviceToHost);
    std::vector<uint32_t> order(G);
    for(uint64_t i = 0; i < G; ++i) order[i] = (uint32_t)i;
    std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return cyc[x] > cyc[y]; });
    double tot = 0; for(uint64_t i = 0; i < G; ++i) tot += cyc[i];
    {
      const uint32_t edges[] = { 1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1024, 1536, 4096, 0xffffffffu };
      uint64_t cntb[19] = { }, hitb[19] = { };
      for(uint64_t i = 0; i < G; ++i) { const uint64_t n = gs[i + 1] - gs[i]; int b = 0; while(n > edges[b]) ++b; cntb[b]++; hitb[b] += n; }
      fprintf(stderr, "[mr]   group sizes (<= edge: groups / hits):");
      for(int b = 0; b < 19; ++b) if(cntb[b]) fprintf(stderr, " %u: %llu / %llu;", edges[b], (unsigned long long)cntb[b], (unsigned long long)hitb[b]);
      fprintf(stderr, "\n");
    }
    fprintf(stderr, "[mr]   chaining cycles: total %.3g; slowest groups (cycles, hits, chain):", tot);
    for(int i = 0; i < 12 && i < (int)G; ++i) { const uint32_t g = order[i]; fprintf(stderr, " (%u, %llu, %u)", cyc[g], (unsigned long long)(gs[g + 1] - gs[g]), nbv[g] & 0x7fffffffu); }
    fprintf(stderr, "\n");
    for(int w = 0; w < 2 && w < (int)G; ++w) {
      const uint32_t g = order[w];
      const uint64_t n = gs[g + 1] - gs[g];
      std::vector<uint64_t> pv(n);
      cudaMemcpy(pv.data(), A.pays + gs[g], n * 8, cudaMemcpyDeviceToHost);
      fprintf(stderr, "[mr]   slow group %u:", g);
      for(uint64_t t = 0; t < n && t < 120; ++t) fprintf(stderr, " %d:%d", (int32_t)(uint32_t)pv[t], (int32_t)(uint32_t)(pv[t] >> 32));
      fprintf(stderr, "\n");
    }
  }
  if(g_chain_trace) {
    uint32_t h[32];
    cudaMemcpy(h, ctr, sizeof h, cudaMemcpyDeviceToHost);
    fprintf(stderr, "[mr]   groups per class:");
    for(int c = 0; c < kClasses; ++c) fprintf(stderr, " %u", h[c]);
    fprintf(stderr, "  very long chains: %u\n", h[28]);
  }
  return MR_OK;
}

// ---------------------------------------------------------------------------------------------
// self test of div_by_count against the hardware's IEEE division (exposed through the C ABI so the
// GPU test-suite can sweep it): values shaped like the least-squares operands (differences of
// offsets, products of offsets minus running means) over every count up to max_n.
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) division_selftest_kernel(uint64_t samples, uint64_t seed, uint32_t max_n,
                                                                 unsigned long long* mismatches) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  unsigned long long bad = 0;
  for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < samples; i += stride) {
    uint64_t z = seed + i * 0x9e3779b97f4a7c15ULL;               // splitmix64
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL; z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL; z ^= z >> 31;
    uint64_t y = z * 0xd1342543de82ef95ULL + 1;
    y = (y ^ (y >> 29)) * 0xbf58476d1ce4e5b9ULL; y ^= y >> 32;
    const uint32_t n = 1 + (uint32_t)(z % max_n);
    const int e = (int)((y >> 56) % 48) - 8;                      // magnitudes 2^-8 .. 2^39
    double x = ldexp((double)(int64_t)(y & 0xfffffffffffffULL) / 4503599627370496.0 + ((y >> 52) & 1 ? 1.0 : 0.0), e);
    if((y >> 53) & 1) x = -x;
    if(((y >> 54) & 3) == 0) x = (double)(int64_t)((y & 0xffffff)) - 8388608.0;   // plain integers too
    const double dn = (double)n;
    const double want = x / dn;
    const double got = div_by_count(x, dn, 1.0 / dn);
    bad += __double_as_longlong(want) != __double_as_longlong(got);
  }
  if(bad) atomicAdd(mismatches, bad);
}
}

extern "C" int mr_selftest_division(mr_context* ctx, uint64_t samples, uint64_t seed, uint32_t max_n, uint64_t* mismatches) {
  if(!ctx || !mismatches || max_n == 0) return MR_EINVAL;
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  dev_buf d;
  MR_TRY(d.ensure(ctx, sizeof(unsigned long long)));
  MR_CUDA(ctx, cudaMemsetAsync(d.p, 0, sizeof(unsigned long long), ctx->stream));
  division_selftest_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(samples, seed, max_n, d.as<unsigned long long>());
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaMemcpyAsync(mismatches, d.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MR_OK;
}

// Pieces of the create_mega_reads record printer that the host formatter (host/host_common.cpp) and the device
// one (records.cu) share, so that both print the same bytes from one implementation:
//  - the integer and fixed-point number formatters of a mega-read line;
//  - the complement table of the unitig sequences;
//  - libstdc++'s std::sort, step for step, for the device (the reference sorts candidates with std::sort, whose
//    order of tied elements is unspecified; reproducing its exact steps reproduces that order).
// Plain C++17 for the host compiler, __host__ __device__ under nvcc.
#pragma once
#include <cstdint>
#include <cstring>

#ifdef __CUDACC__
#define MR_HD __host__ __device__ __forceinline__
#else
#define MR_HD inline
#endif

namespace mrfmt {

// complement of a unitig base as print_sequence writes an 'R' unitig (super_read_name.cc:106-114): ACGT in either
// case, anything else 'N'
MR_HD char revcomp_base(unsigned char c) {
  switch(c) {
  case 'a': case 'A': return 'T';
  case 'c': case 'C': return 'G';
  case 'g': case 'G': return 'C';
  case 't': case 'T': return 'A';
  default: return 'N';
  }
}

MR_HD int fmt_uint(char* p, uint64_t v) {
  int n = 1;
  for(uint64_t t = v; t >= 10; t /= 10) ++n;
  for(int i = n - 1; i >= 0; --i) { p[i] = (char)('0' + v % 10); v /= 10; }
  return n;
}
MR_HD int fmt_int(char* p, int64_t v) {
  if(v < 0) { *p = '-'; return 1 + fmt_uint(p + 1, (uint64_t)0 - (uint64_t)v); }
  return fmt_uint(p, (uint64_t)v);
}
MR_HD int fmt_u128(char* p, unsigned __int128 v) {
  if((v >> 64) == 0) return fmt_uint(p, (uint64_t)v);
  char t[40];
  int n = 0;
  while(v) { t[n++] = (char)('0' + (int)(v % 10)); v /= 10; }
  for(int i = 0; i < n; ++i) p[i] = t[n - 1 - i];
  return n;
}

// Longest text fmt_fixed writes: sign, 309 integer digits, point, 4 decimals.
constexpr int kFixedMax = 320;

// Exactly what glibc's printf("%.<d>f", x) prints, d = 2 or 4, for every double.  x = m 2^e exactly; below 2^64
// the scaled value m 10^d 2^e is a 128-bit integer product rounded once at the binary point, ties to even (the
// rounding printf applies to the exact value).  From 2^64 on x is an integer, printed from a multi-word binary
// number, followed by d zeros.  inf and nan print as glibc prints them, with the sign of x.
MR_HD int fmt_fixed(char* p, double x, int d) {
  uint64_t bits;
  memcpy(&bits, &x, sizeof bits);
  const int ex = (int)((bits >> 52) & 0x7ff);
  uint64_t m = bits & ((1ULL << 52) - 1);
  char* q = p;
  if(bits >> 63) *q++ = '-';
  if(ex == 0x7ff) {
    if(m) { q[0] = 'n'; q[1] = 'a'; q[2] = 'n'; } else { q[0] = 'i'; q[1] = 'n'; q[2] = 'f'; }
    return (int)(q + 3 - p);
  }
  int e;
  if(ex == 0) e = -1074; else { m |= 1ULL << 52; e = ex - 1075; }
  const uint32_t scale = d == 2 ? 100u : 10000u;
  if(e <= 11) {                                            // |x| < 2^64
    const unsigned __int128 P = (unsigned __int128)m * scale;     // < 2^67
    unsigned __int128 n = 0;
    if(e >= 0) n = P << e;
    else if(-e < 100) {                                    // else P 2^e < 2^-33: rounds to 0
      const int s = -e;
      n = P >> s;
      const unsigned __int128 rem = P - (n << s), half = (unsigned __int128)1 << (s - 1);
      if(rem > half || (rem == half && (n & 1))) ++n;
    }
    uint32_t f;
    if((n >> 64) == 0) {                                   // the common case, in 64-bit arithmetic
      const uint64_t n64 = (uint64_t)n;
      q += fmt_uint(q, n64 / scale);
      f = (uint32_t)(n64 % scale);
    } else {
      q += fmt_u128(q, n / scale);
      f = (uint32_t)(n % scale);
    }
    *q++ = '.';
    for(int i = d - 1; i >= 0; --i) { q[i] = (char)('0' + f % 10); f /= 10; }
    return (int)(q + d - p);
  }
  // |x| >= 2^64: the integer m 2^e in 32-bit words, least significant first (e <= 971: at most 1024 bits)
  uint32_t w[34];
  for(int i = 0; i < 34; ++i) w[i] = 0;
  const int wi = e >> 5, sh = e & 31;
  const unsigned __int128 mm = (unsigned __int128)m << sh;
  w[wi] = (uint32_t)mm; w[wi + 1] = (uint32_t)(mm >> 32); w[wi + 2] = (uint32_t)(mm >> 64);
  int top = wi + 2;
  uint32_t chunk[36];                                       // base-10^9 digits, least significant first
  int nc = 0;
  while(top >= 0) {
    uint64_t rem = 0;
    for(int i = top; i >= 0; --i) {
      const uint64_t cur = (rem << 32) | w[i];
      w[i] = (uint32_t)(cur / 1000000000u);
      rem = cur % 1000000000u;
    }
    chunk[nc++] = (uint32_t)rem;
    while(top >= 0 && w[top] == 0) --top;
  }
  q += fmt_uint(q, chunk[nc - 1]);
  for(int c = nc - 2; c >= 0; --c) {
    uint32_t v = chunk[c];
    for(int i = 8; i >= 0; --i) { q[i] = (char)('0' + v % 10); v /= 10; }
    q += 9;
  }
  *q++ = '.';
  for(int i = 0; i < d; ++i) *q++ = '0';
  return (int)(q - p);
}

// ---- "%g": what glibc's printf("%g", x) prints (precision 6), the default ostream output of a double that
// jf_aligner's coords lines use for stretch, offset and avg_err (jf_aligner.cc:58).  x = m 2^e exactly is rounded
// once to 6 significant digits D 10^(X-5), ties to even, X taken after the rounding (999999.5 -> 1e+06); then
// fixed notation for -4 <= X < 6, else d.ddddde+XX, trailing zeros and a bare point dropped.
// Longest text: "-1.23457e-308".
constexpr int kGeneralMax = 16;

namespace detail {
MR_HD int ndigits(uint64_t v) { int n = 1; while(v >= 10) { v /= 10; ++n; } return n; }
MR_HD uint64_t pow10u(int s) { uint64_t p = 1; while(s-- > 0) p *= 10; return p; }

// 2^-16 <= x < 2^64 (2^52 <= m < 2^53, -68 <= e <= 11): 64- and 128-bit integers, no division wider than 64 bits
MR_HD void general_digits(uint64_t m, int e, uint32_t& D, int& X) {
  const int q = -e;
  const uint64_t I = e >= 0 ? m << e : (q < 64 ? m >> q : 0);     // floor(x)
  uint64_t d;
  bool up;
  if(I >= 100000) {                                      // X >= 5: X is the integer part's digit count - 1
    X = ndigits(I) - 1;
    const uint64_t pw = pow10u(X - 5);
    d = I / pw;
    const uint64_t r = I % pw;
    const uint64_t f = e < 0 ? m & ((1ULL << q) - 1) : 0;   // fraction bits (x >= 2^16: q <= 36)
    if(pw == 1) up = e < 0 && (f > (1ULL << (q - 1)) || (f == (1ULL << (q - 1)) && (d & 1)));
    else { const uint64_t h = pw / 2; up = r > h || (r == h && (f != 0 || (d & 1))); }   // r + fraction against pw / 2
  } else {                                               // x < 10^5, so e < 0: D = round(m 10^(5 - X) 2^e)
    const uint64_t w = (uint64_t)(((unsigned __int128)m * 100000u) >> q);   // floor(x 10^5) >= 1
    X = ndigits(w) - 6;
    const unsigned __int128 P = (unsigned __int128)m * pow10u(5 - X);         // < 2^87
    d = (uint64_t)(P >> q);
    const unsigned __int128 rem = P - ((unsigned __int128)d << q), half = (unsigned __int128)1 << (q - 1);
    up = rem > half || (rem == half && (d & 1));
  }
  D = (uint32_t)(d + up);
}

// multi-word integers for the rest of the double range: 40 32-bit words, least significant first.  The loops stay
// rolled on the device: unrolled, the words went to registers, and the callers took on the callee's 150 registers.
#ifdef __CUDA_ARCH__
#define MR_ROLLED _Pragma("unroll 1")
#else
#define MR_ROLLED
#endif
constexpr int kBigWords = 40;
MR_HD void big_mul(uint32_t* a, uint32_t f) {
  uint64_t c = 0;
  MR_ROLLED for(int i = 0; i < kBigWords; ++i) { const uint64_t t = (uint64_t)a[i] * f + c; a[i] = (uint32_t)t; c = t >> 32; }
}
MR_HD void big_shl(uint32_t* a, int s) {
  const int ws = s >> 5, bs = s & 31;
  MR_ROLLED for(int i = kBigWords - 1; i >= 0; --i) {
    const uint32_t hi = i - ws >= 0 ? a[i - ws] : 0, lo = i - ws - 1 >= 0 ? a[i - ws - 1] : 0;
    a[i] = bs ? (hi << bs) | (lo >> (32 - bs)) : hi;
  }
}
MR_HD void big_shr1(uint32_t* a) {
  MR_ROLLED for(int i = 0; i < kBigWords; ++i) a[i] = (a[i] >> 1) | (i + 1 < kBigWords ? a[i + 1] << 31 : 0);
}
MR_HD int big_cmp(const uint32_t* a, const uint32_t* b) {
  MR_ROLLED for(int i = kBigWords - 1; i >= 0; --i) if(a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
  return 0;
}
MR_HD void big_sub(uint32_t* a, const uint32_t* b) {
  int64_t br = 0;
  MR_ROLLED for(int i = 0; i < kBigWords; ++i) { const int64_t t = (int64_t)a[i] - b[i] - br; a[i] = (uint32_t)t; br = t < 0; }
}

// any finite x = m 2^e > 0 (subnormals included): D = round(num / den) with num = m 2^max(e, 0) 10^max(5 - X, 0) and
// den = 2^max(-e, 0) 10^max(X - 5, 0) (at most 1146 bits), X found from an estimate by checking 10^5 <= D < 10^6.
// Kept out of line: the coords never reach it, and its 320 bytes of words stay out of the callers' frames.
#ifdef __CUDACC__
__host__ __device__ __noinline__ inline
#else
__attribute__((noinline)) inline
#endif
void general_digits_big(uint64_t m, int e, uint32_t& D, int& X) {
  int b = e + 63;                                        // floor(log2 x)
  for(uint64_t t = m; !(t >> 63); t <<= 1) --b;
  X = (int)((double)b * 0.30102999566398120);            // within one of floor(log10 x)
  uint32_t num[kBigWords], den[kBigWords];
  for(;;) {
    MR_ROLLED for(int i = 0; i < kBigWords; ++i) num[i] = den[i] = 0;
    num[0] = (uint32_t)m; num[1] = (uint32_t)(m >> 32); den[0] = 1;
    if(e > 0) big_shl(num, e); else big_shl(den, -e);
    for(int s = X - 5; s < 0; ++s) big_mul(num, 10);
    for(int s = X - 5; s > 0; --s) big_mul(den, 10);
    big_shl(den, 24);                                    // the quotient is below 10^7 < 2^25: restoring division
    uint32_t d = 0;
    for(int bit = 24; bit >= 0; --bit) {
      if(big_cmp(num, den) >= 0) { big_sub(num, den); d |= 1u << bit; }
      if(bit) big_shr1(den);
    }
    if(d >= 1000000) { ++X; continue; }
    if(d < 100000) { --X; continue; }
    big_shl(num, 1);                                     // the remainder against den / 2
    const int c = big_cmp(num, den);
    D = d + (c > 0 || (c == 0 && (d & 1)));
    return;
  }
}

MR_HD int general_text(char* p, bool neg, uint32_t D, int X) {
  char d[6];
  for(int i = 5; i >= 0; --i) { d[i] = (char)('0' + D % 10); D /= 10; }
  int nd = 6;                                            // digits left once the trailing zeros are gone
  while(nd > 1 && d[nd - 1] == '0') --nd;
  char* q = p;
  if(neg) *q++ = '-';
  if(X >= -4 && X < 6) {
    if(X >= 0) {
      for(int i = 0; i <= X; ++i) *q++ = d[i];
      if(nd > X + 1) { *q++ = '.'; for(int i = X + 1; i < nd; ++i) *q++ = d[i]; }
    } else {
      *q++ = '0'; *q++ = '.';
      for(int i = 0; i < -X - 1; ++i) *q++ = '0';
      for(int i = 0; i < nd; ++i) *q++ = d[i];
    }
  } else {
    *q++ = d[0];
    if(nd > 1) { *q++ = '.'; for(int i = 1; i < nd; ++i) *q++ = d[i]; }
    *q++ = 'e';
    *q++ = X < 0 ? '-' : '+';
    const int ax = X < 0 ? -X : X;
    if(ax < 10) *q++ = '0';
    q += fmt_uint(q, (uint64_t)ax);
  }
  return (int)(q - p);
}
} // namespace detail

MR_HD int fmt_general(char* p, double x) {
  uint64_t bits;
  memcpy(&bits, &x, sizeof bits);
  const bool neg = bits >> 63;
  const int ex = (int)((bits >> 52) & 0x7ff);
  const uint64_t m = bits & ((1ULL << 52) - 1);
  if(ex == 0x7ff || (ex == 0 && m == 0)) {
    char* q = p;
    if(neg) *q++ = '-';
    if(ex == 0) { *q++ = '0'; return (int)(q - p); }
    if(m) { q[0] = 'n'; q[1] = 'a'; q[2] = 'n'; } else { q[0] = 'i'; q[1] = 'n'; q[2] = 'f'; }
    return (int)(q + 3 - p);
  }
  uint32_t D;
  int X;
  if(ex >= 1023 - 16 && ex < 1023 + 64) detail::general_digits(m | (1ULL << 52), ex - 1075, D, X);
  else detail::general_digits_big(ex ? m | (1ULL << 52) : m, ex ? ex - 1075 : -1074, D, X);
  if(D == 1000000) { D = 100000; ++X; }
  return detail::general_text(p, neg, D, X);
}

// ---- std::sort of libstdc++ (bits/stl_algo.h, bits/stl_heap.h): introsort with threshold 16 and depth limit
// 2 floor(log2 n), median of three on first + 1, mid, last - 1 moved to first, unguarded partition, heap sort when
// the depth runs out, then __final_insertion_sort.  Sorts a[0, n) of int with comp(x, y) meaning "x before y".
// The recursion on the right part becomes an explicit stack (the parts are disjoint, so the order in which they
// are processed does not change the result).  The unguarded scans are bounded by the array: for a comparator that
// is a strict weak order the bounds are never reached, exactly as in libstdc++.
namespace detail {
template<class Comp> MR_HD void adjust_heap(int* a, long hole, long len, int value, Comp& comp) {
  const long top = hole;
  long second = hole;
  while(second < (len - 1) / 2) {
    second = 2 * (second + 1);
    if(comp(a[second], a[second - 1])) --second;
    a[hole] = a[second];
    hole = second;
  }
  if((len & 1) == 0 && second == (len - 2) / 2) {
    second = 2 * (second + 1);
    a[hole] = a[second - 1];
    hole = second - 1;
  }
  long parent = (hole - 1) / 2;
  while(hole > top && comp(a[parent], value)) {
    a[hole] = a[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  a[hole] = value;
}
template<class Comp> MR_HD void heap_sort(int* a, long len, Comp& comp) {
  if(len >= 2)
    for(long parent = (len - 2) / 2; ; --parent) {
      adjust_heap(a, parent, len, a[parent], comp);
      if(parent == 0) break;
    }
  for(long last = len - 1; last > 0; --last) {
    const int v = a[last];
    a[last] = a[0];
    adjust_heap(a, 0, last, v, comp);
  }
}
template<class Comp> MR_HD void linear_insert(int* a, long i, long lo, Comp& comp) {
  const int v = a[i];
  long j = i - 1;
  while(j >= lo && comp(v, a[j])) { a[j + 1] = a[j]; --j; }
  a[j + 1] = v;
}
} // namespace detail

template<class Comp> MR_HD void std_sort(int* a, long n, Comp comp) {
  if(n <= 1) return;
  int lg = 0;
  for(long t = n; t > 1; t >>= 1) ++lg;
  struct range { long lo, hi; int depth; };
  range stack[130];
  int sp = 0;
  stack[sp++] = range{ 0, n, 2 * lg };
  while(sp) {
    range rg = stack[--sp];
    long lo = rg.lo, hi = rg.hi;
    int depth = rg.depth;
    while(hi - lo > 16) {
      if(depth == 0) { detail::heap_sort(a + lo, hi - lo, comp); break; }
      --depth;
      // __move_median_to_first(lo, lo + 1, mid, hi - 1)
      const long mid = lo + (hi - lo) / 2, x = lo + 1, z = hi - 1;
      long pick;
      if(comp(a[x], a[mid])) {
        if(comp(a[mid], a[z])) pick = mid; else if(comp(a[x], a[z])) pick = z; else pick = x;
      } else if(comp(a[x], a[z])) pick = x;
      else if(comp(a[mid], a[z])) pick = z;
      else pick = mid;
      { const int t = a[lo]; a[lo] = a[pick]; a[pick] = t; }
      // __unguarded_partition(lo + 1, hi, pivot = lo)
      long f = lo + 1, l = hi;
      while(true) {
        while(f < hi && comp(a[f], a[lo])) ++f;
        --l;
        while(l > lo && comp(a[lo], a[l])) --l;
        if(!(f < l)) break;
        const int t = a[f]; a[f] = a[l]; a[l] = t;
        ++f;
      }
      stack[sp++] = range{ f, hi, depth };
      hi = f;
    }
  }
  // __final_insertion_sort
  const long head = n > 16 ? 16 : n;
  for(long i = 1; i < head; ++i) {
    if(comp(a[i], a[0])) {
      const int v = a[i];
      for(long j = i; j > 0; --j) a[j] = a[j - 1];
      a[0] = v;
    } else detail::linear_insert(a, i, 0, comp);
  }
  for(long i = head; i < n; ++i) detail::linear_insert(a, i, 0, comp);
}

} // namespace mrfmt

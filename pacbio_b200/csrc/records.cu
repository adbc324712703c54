// Mega-read records on the device: the printing side of overlap_graph (overlap_graph.cc:61-299,
// overlap_graph.hpp:198-262) over the rows and graph nodes a batch left in the context's workspace.
//  1. plan: per read, the best end node of every component (root order), --trim match, the density / length
//     filters and the tiling; the lines of the read are the candidates in print order.  A thread per read, a warp
//     per read with many rows (the overlap and containment scans of the greedy tiling spread over its lanes).
//  2. measure: per line, its byte length (numbers, the spliced path's name, sr_len, the sequence), the first line
//     of a read also counting the read's header; an exclusive scan places every line.
//  3. emit: a warp per line writes it; the sequence pieces are copied by all lanes, complemented on the fly for
//     'R' unitigs.
// The text is copied into a pooled pinned slab.  The formatters and the std::sort port are records_common.hpp,
// shared with the host formatter (host/host_common.cpp), which prints the same bytes.
#include "align.cuh"
#include "records_common.hpp"

#include <cstring>
#include <memory>

struct mr_unitigs {
  int device = 0;
  uint32_t n = 0;
  dev_buf seq, off;
};

namespace {

// one candidate mega-read (overlap_graph.hpp:51-63), stored at the row of its end node
struct cand_t {
  double imp_s, imp_e, tiling_start, tiling_end, density;
  int32_t start_node, end_node, start_unitig, start_offset, end_offset, nb_unitigs;
  int32_t ok;                                   // an end node that passes the density and length filters
  int32_t pad;
};
struct tinfo_t { double pos; int32_t score, node, previous, length; };

// what the measure pass learns about a line and the emit pass needs again (stored per line, so that emit walks the
// path only to write it)
struct line_info {
  uint64_t pb, pe, first, qe_out;
  uint32_t hdr, num_len, name_len;
  int32_t sr_len;
};

struct rec_args {
  graph_args g;                                 // the rows and nodes (align.cuh)
  uint32_t nreads;
  int32_t k;
  double overlap_play, density, min_length;
  int tiling, trim, big_rows;
  // per row
  cand_t* cand;
  int32_t *comp_slot, *comp_best, *mrs, *sort_t, *tiled, *order;
  double* weight;
  double2 *cov, *placed;
  tinfo_t* info;
  // per read
  uint32_t* nlines;
  uint64_t* line_base;
  // per line (at most one per row)
  uint32_t* line_read;
  int32_t*  line_node;
  uint32_t* line_len;
  uint64_t* line_off;
  line_info* line_inf;
  const uint64_t* n_lines;                      // device: total lines
  // text
  const char* useq; const uint64_t* uoff; uint32_t nu;
  const char* names; const uint64_t* name_off;
  char* text;
  uint64_t text_size;
  unsigned long long* err;                      // smallest (read << 1 | kind) that failed, see kErr*
};
constexpr unsigned long long kErrRoot = 0, kErrUnitig = 1;   // the component check comes before the read's printing

__device__ __forceinline__ void record_error(const rec_args& A, uint32_t r, unsigned long long kind) {
  atomicMin(A.err, ((unsigned long long)r << 1) | kind);
}

// ---- group helpers: W = 1 (a thread) or 32 (a warp); every lane holds the same uniform state --------------------
template<int W> __device__ __forceinline__ void gsync() { if(W > 1) __syncwarp(); }
template<int W> __device__ __forceinline__ bool gany(bool x) { return W > 1 ? __any_sync(MR_FULL_MASK, x) : x; }
template<int W> __device__ __forceinline__ int gsum(int x) {
  if(W > 1) for(int o = 16; o; o >>= 1) x += __shfl_xor_sync(MR_FULL_MASK, x, o);
  return x;
}
template<int W> __device__ __forceinline__ int gbcast(int x) { return W > 1 ? __shfl_sync(MR_FULL_MASK, x, 0) : x; }
// std::min / std::max of the joined interval set (boost::icl through tile_greedy's use of it)
__device__ __forceinline__ double dmin(double a, double b) { return b < a ? b : a; }
__device__ __forceinline__ double dmax(double a, double b) { return a < b ? b : a; }
template<int W> __device__ __forceinline__ double gmin(double x) {
  if(W > 1) for(int o = 16; o; o >>= 1) x = dmin(x, __shfl_xor_sync(MR_FULL_MASK, x, o));
  return x;
}
template<int W> __device__ __forceinline__ double gmax(double x) {
  if(W > 1) for(int o = 16; o; o >>= 1) x = dmax(x, __shfl_xor_sync(MR_FULL_MASK, x, o));
  return x;
}

// unitig path of a row's super-read in the orientation the row uses it (super_reads::path_at)
__device__ __forceinline__ uint32_t path_len(const graph_args& g, uint64_t row) {
  const uint32_t s = g.c.sr[row];
  return (uint32_t)(g.unitig_off[s + 1] - g.unitig_off[s]);
}
__device__ __forceinline__ uint32_t path_at(const graph_args& g, uint64_t row, uint32_t t) {
  const uint32_t s = g.c.sr[row];
  const uint64_t b = g.unitig_off[s], e = g.unitig_off[s + 1];
  return g.c.use_bwd[row] ? (g.unitig_ids[e - 1 - t] ^ 1u) : g.unitig_ids[b + t];
}
__device__ __forceinline__ int ulen_of(const graph_args& g, uint32_t id) { return id < g.n_unitigs ? g.unitig_len[id] : 0; }

// candidate of row i of a read (mega_reads_per_comp and trim_match, overlap_graph.cc:78-161)
__device__ void make_candidate(const rec_args& A, uint64_t b, int i, double pb_size, cand_t& mr) {
  const graph_args& g = A.g;
  const uint64_t row = b + i;
  mr.start_node = g.lstart[row] == -1 ? i : g.lstart[row];
  mr.end_node = i;
  const uint64_t srow = b + mr.start_node;
  mr.start_unitig = 0;
  mr.nb_unitigs = g.lunitigs[row];
  mr.imp_s = g.c.stretch[srow] + g.c.offset[srow];
  { const double t = g.c.stretch[row] * (double)g.c.ql[row]; mr.imp_e = t + g.c.offset[row]; }
  mr.tiling_start = g.c.rs[srow];
  mr.tiling_end = g.c.re[row];
  mr.start_offset = mr.end_offset = 0;
  auto unitig_id = [&](uint64_t r, uint32_t t) -> uint32_t { return t < path_len(g, r) ? (path_at(g, r, t) >> 1) : 0x7fffffffu; };
  if(A.trim) {
    const double node_imp_s = g.c.stretch[srow] + g.c.offset[srow];
    if(node_imp_s < 1) {
      const int32_t* ki = g.kinfo + g.c.info_off[srow];
      const int ilen = (int)g.c.info_len[srow];
      int offset = 0, su;
      for(su = 0; su < ilen; su += 2) {
        if(ki[su]) break;
        offset += ulen_of(g, unitig_id(srow, su / 2));
      }
      su /= 2;
      mr.start_unitig = su;
      mr.nb_unitigs -= su;
      offset -= (A.k - 1) * su;
      mr.start_offset = offset;
      { const double t = g.c.stretch[srow] * (double)(offset + 1); mr.imp_s = t + g.c.offset[srow]; }
    }
    if(mr.imp_e > (double)g.c.ql[row]) {
      const int32_t* ki = g.kinfo + g.c.info_off[row];
      const int ilen = (int)g.c.info_len[row];
      int offset = 0, eu;
      for(eu = ilen - 1; eu >= 0; eu -= 2) {
        if(ki[eu]) break;
        offset += ulen_of(g, unitig_id(row, eu / 2));
      }
      eu /= 2;
      const int removed = ilen / 2 - eu;
      mr.nb_unitigs -= removed;
      offset -= (A.k - 1) * removed;
      mr.end_offset = offset;
      { const double t = g.c.stretch[row] * (double)((int64_t)g.c.ql[row] - offset); mr.imp_e = t + g.c.offset[row]; }
    }
  }
  const double len = dmin(pb_size + 0.5, mr.tiling_end) - dmax(0.5, mr.tiling_start);
  mr.density = (double)g.lpath[row] / len;
  mr.ok = g.end_node[row] && !(mr.density < A.density) && !((mr.tiling_end - mr.tiling_start) < A.min_length);
}

// The lines of read r, in print order: order[b + j] is the end node of line j, nlines[r] their number.
template<int W>
__device__ void plan_read(const rec_args& A, uint32_t r, int lane) {
  const graph_args& g = A.g;
  const uint64_t b = g.read_coords[r];
  const int n = (int)(g.read_coords[r + 1] - b);
  if(n == 0) { if(lane == 0) A.nlines[r] = 0; return; }
  const double pb_size = (double)g.read_len[r];
  for(int i = lane; i < n; i += W) {
    cand_t mr;
    make_candidate(A, b, i, pb_size, mr);
    A.cand[b + i] = mr;
    A.comp_slot[b + i] = -1;
  }
  gsync<W>();
  // the best candidate of every component (a later one replaces it only when strictly better), then the
  // components in increasing root order
  int ncomp = 0;
  if(lane == 0) {
    int nslots = 0;
    for(int i = 0; i < n; ++i) {
      const cand_t& c = A.cand[b + i];
      if(!c.ok) continue;
      const int root = g.component[b + i];
      if(root < 0 || root >= n) { record_error(A, r, kErrRoot); continue; }
      const int slot = A.comp_slot[b + root];
      if(slot < 0) { A.comp_slot[b + root] = nslots; A.comp_best[b + nslots] = i; ++nslots; }
      else {
        const int cur = A.comp_best[b + slot];
        const int olpath = g.lpath[b + cur];
        if(g.lpath[b + i] > olpath || (g.lpath[b + i] == olpath && c.density > A.cand[b + cur].density)) A.comp_best[b + slot] = i;
      }
    }
    for(int root = 0; root < n && ncomp < nslots; ++root) {
      const int slot = A.comp_slot[b + root];
      if(slot >= 0) { A.mrs[b + ncomp] = A.comp_best[b + slot]; A.sort_t[b + ncomp] = ncomp; ++ncomp; }
    }
  }
  ncomp = gbcast<W>(ncomp);
  gsync<W>();
  if(ncomp == 0) { if(lane == 0) A.nlines[r] = 0; return; }
  const cand_t* cand = A.cand + b;
  const int32_t* mrs = A.mrs + b;
  int32_t* sort_t = A.sort_t + b;
  int32_t* tiled = A.tiled + b;
  auto lpath_of = [&](int m) { return g.lpath[b + mrs[m]]; };
  auto by_pos = [&](int i, int j) {
    const cand_t& x = cand[mrs[i]]; const cand_t& y = cand[mrs[j]];
    return x.imp_s < y.imp_s || (x.imp_s == y.imp_s && x.imp_e < y.imp_e);
  };
  const double K = A.k;
  int ntiled = 0;
  // tile_greedy (overlap_graph.cc:165-197) over the candidates in sort_t order
  auto greedy = [&]() {
    double2* cov = A.cov + b;
    double2* placed = A.placed + b;
    int ncov = 0, nplaced = 0;
    for(int t = 0; t < ncomp; ++t) {
      const int m = sort_t[t];
      const cand_t& c = cand[mrs[m]];
      const double lo = c.tiling_start, up = c.tiling_end;
      const double plen = lo < up ? up - lo : 0.0;
      const double max_overlap = dmax(K * A.overlap_play, plen * (A.overlap_play - 0.9));
      bool hit = false;
      for(int j = lane; j < ncov; j += W) {
        const double2 y = cov[j];
        const double l = dmax(y.x, lo), u = dmin(y.y, up);
        if(l < u && u - l >= max_overlap) hit = true;
      }
      if(gany<W>(hit)) continue;
      bool contained = false;
      for(int j = lane; j < nplaced; j += W) {
        const double2 p = placed[j];
        if(!(lo < up) || (p.x <= lo && up <= p.y)) contained = true;
      }
      if(gany<W>(contained)) continue;
      if(lo < up) {                                 // joined_set::add: merge the spans that touch [lo, up)
        int before = 0, after = 0;
        double nlo = lo, nup = up;
        for(int j = lane; j < ncov; j += W) {
          const double2 y = cov[j];
          if(y.y < lo) ++before;
          else if(up < y.x) ++after;
          else { nlo = dmin(nlo, y.x); nup = dmax(nup, y.y); }
        }
        before = gsum<W>(before); after = gsum<W>(after);
        nlo = gmin<W>(nlo); nup = gmax<W>(nup);
        const int middle = ncov - before - after, delta = 1 - middle, from = ncov - after;
        if(delta < 0) {                             // the spans behind move towards the front
          for(int base = from; base < ncov; base += W) {
            const int j = base + lane;
            double2 y;
            if(j < ncov) y = cov[j];
            gsync<W>();
            if(j < ncov) cov[j + delta] = y;
            gsync<W>();
          }
        } else if(delta > 0) {                      // one place further back, last first
          for(int base = ncov - W; base > from - W; base -= W) {
            const int j = base + lane;
            double2 y;
            const bool in = j >= from && j < ncov;
            if(in) y = cov[j];
            gsync<W>();
            if(in) cov[j + 1] = y;
            gsync<W>();
          }
        }
        if(lane == 0) cov[before] = make_double2(nlo, nup);
        ncov += delta;
      }
      if(lane == 0) { placed[nplaced] = make_double2(lo, up); tiled[ntiled] = m; }
      ++nplaced; ++ntiled;
      gsync<W>();
    }
  };
  // the std::sort calls are the reference's own (same comparator, same input order): their order on ties too
  switch(A.tiling) {
  case 1:
    if(lane == 0) mrfmt::std_sort(sort_t, ncomp, [&](int i, int j) { return lpath_of(j) < lpath_of(i); });
    gsync<W>();
    greedy();
    if(lane == 0) mrfmt::std_sort(tiled, ntiled, by_pos);
    break;
  case 3: {
    double* w = A.weight + b;
    for(int i = lane; i < ncomp; i += W) {
      const cand_t& c = cand[mrs[i]];
      const double d2 = c.density * c.density;
      w[i] = d2 * (double)(g.c.re[b + c.end_node] - g.c.rs[b + c.start_node] + 1);
    }
    gsync<W>();
    if(lane == 0) mrfmt::std_sort(sort_t, ncomp, [&](int i, int j) { return w[j] < w[i]; });
    gsync<W>();
    greedy();
    if(lane == 0) mrfmt::std_sort(tiled, ntiled, by_pos);
    break;
  }
  case 2:                                           // tile_maximal (overlap_graph.cc:212-252)
    if(lane == 0) {
      mrfmt::std_sort(sort_t, ncomp, [&](int i, int j) { return cand[mrs[i]].tiling_end < cand[mrs[j]].tiling_end; });
      tinfo_t* info = A.info + b;
      int ninfo = 0;
      { const int m = sort_t[0]; info[ninfo++] = tinfo_t{ cand[mrs[m]].tiling_end, lpath_of(m), m, -1, 1 }; }
      for(int t = 1; t < ncomp; ++t) {
        const int m = sort_t[t];
        const double lstart = cand[mrs[m]].tiling_start;
        const double key = dmin(lstart + K * A.overlap_play, cand[mrs[m]].tiling_end);
        int lo = 0, len = ninfo;                    // std::upper_bound
        while(len > 0) {
          const int half = len >> 1;
          if(key < info[lo + half].pos) len = half;
          else { lo += half + 1; len -= half + 1; }
        }
        int i = lo - 1;
        while(i >= 0 && cand[mrs[info[i].node]].tiling_start >= lstart) i = info[i].previous;
        const int nscore = (i >= 0 ? info[i].score : 0) + lpath_of(m);
        if(nscore > info[ninfo - 1].score) info[ninfo++] = tinfo_t{ cand[mrs[m]].tiling_end, nscore, m, i, (i >= 0 ? info[i].length : 0) + 1 };
      }
      ntiled = info[ninfo - 1].length;
      int ptr = ninfo - 1;
      for(int t = ntiled - 1; t >= 0; --t) { tiled[t] = info[ptr].node; ptr = info[ptr].previous; }
      mrfmt::std_sort(tiled, ntiled, by_pos);
    }
    ntiled = gbcast<W>(ntiled);
    break;
  default: break;
  }
  gsync<W>();
  const int32_t* fin = ntiled ? tiled : sort_t;
  const int nl = ntiled ? ntiled : ncomp;
  for(int j = lane; j < nl; j += W) A.order[b + j] = mrs[fin[j]];
  if(lane == 0) A.nlines[r] = (uint32_t)nl;
}

__global__ void plan_small_kernel(rec_args A) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if(r >= A.nreads) return;
  if(A.g.read_coords[r + 1] - A.g.read_coords[r] > (uint64_t)A.big_rows) return;
  plan_read<1>(A, r, 0);
}
__global__ void plan_big_kernel(rec_args A) {
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if(r >= A.nreads) return;
  if(A.g.read_coords[r + 1] - A.g.read_coords[r] <= (uint64_t)A.big_rows) return;
  plan_read<32>(A, r, (int)lane_id());
}

__global__ void expand_lines_kernel(rec_args A) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if(r >= A.nreads) return;
  const uint64_t b = A.g.read_coords[r], l0 = A.line_base[r];
  const uint32_t nl = A.nlines[r];
  for(uint32_t j = 0; j < nl; ++j) { A.line_read[l0 + j] = r; A.line_node[l0 + j] = A.order[b + j]; }
}

// ---- one line (print_mega_reads, overlap_graph.cc:254-299) ---------------------------------------------------------
// The path of a line is spliced from the end node back along lprev: every node prepends a piece of its super-read's
// path.  Entries [0, first) that no node fills stay 0 ("0F").  walk() hands each filled entry to f(index, entry),
// pieces from the back of the path to its front, and returns `first`.
template<class F>
__device__ uint64_t walk_path(const graph_args& g, uint64_t b, int end_node, uint64_t P, F&& f) {
  auto prepend = [&](uint64_t offset, uint64_t row, uint64_t last) -> uint64_t {
    const uint64_t sz = path_len(g, row);
    if(0 >= sz) return offset;
    const uint64_t to_copy = (last < sz - 1 ? last : sz - 1) + 1;
    if(to_copy > offset) return offset;
    for(uint64_t t = to_copy; t-- > 0;) f(offset - to_copy + t, path_at(g, row, (uint32_t)t));
    return offset - to_copy;
  };
  const uint64_t erow = b + end_node;
  uint64_t offset = prepend(P, erow, (uint64_t)path_len(g, erow) - 1);
  int node_j = end_node, node_i = g.lprev[erow];
  while(node_i >= 0) {
    const uint64_t irow = b + node_i, jrow = b + node_j;
    const uint64_t overlap = (uint64_t)(int64_t)g.lunitigs[irow] + path_len(g, jrow) - (uint64_t)(int64_t)g.lunitigs[jrow];
    offset = prepend(offset, irow, (uint64_t)path_len(g, irow) - 1 - overlap);
    node_j = node_i;
    node_i = g.lprev[irow];
  }
  return offset;
}

struct line_t {
  uint32_t r;
  uint64_t b, erow, srow, P, first;
  const cand_t* c;
  uint32_t hdr, num_len, name_len, sr_digits;
  int32_t sr_len;
  uint64_t pb, pe, seq_len, qe_out;
  uint32_t len;
  bool bad_unitig;
};


__device__ __forceinline__ uint32_t ndigits(uint64_t v) { uint32_t n = 1; while(v >= 10) { v /= 10; ++n; } return n; }

// number columns "%.2f %.2f %d %d %d %llu %d %.4f " (overlap_graph.cc:285-290)
__device__ int write_numbers(const rec_args& A, const line_t& L, char* w) {
  const graph_args& g = A.g;
  char* p = w;
  p += mrfmt::fmt_fixed(p, L.c->imp_s, 2); *p++ = ' ';
  p += mrfmt::fmt_fixed(p, L.c->imp_e, 2); *p++ = ' ';
  p += mrfmt::fmt_int(p, g.c.rs[L.srow]); *p++ = ' ';
  p += mrfmt::fmt_int(p, g.c.re[L.erow]); *p++ = ' ';
  p += mrfmt::fmt_int(p, g.c.qs[L.srow] - L.c->start_offset); *p++ = ' ';
  p += mrfmt::fmt_uint(p, L.qe_out); *p++ = ' ';
  p += mrfmt::fmt_int(p, g.lpath[L.erow]); *p++ = ' ';
  p += mrfmt::fmt_fixed(p, L.c->density, 4); *p++ = ' ';
  return (int)(p - w);
}

__device__ __forceinline__ void line_rows(const rec_args& A, uint64_t l, line_t& L);

__device__ void layout_line(const rec_args& A, uint64_t l, line_t& L) {
  const graph_args& g = A.g;
  line_rows(A, l, L);
  const cand_t& c = *L.c;
  L.hdr = l == A.line_base[L.r] ? (uint32_t)(A.name_off[L.r + 1] - A.name_off[L.r]) + 2 : 0;
  // path name, sr_len and the sequence's length in one pass over the filled entries; the unfilled ones are id 0
  const int64_t su = c.start_unitig, se = (int64_t)c.start_unitig + c.nb_unitigs;
  L.pb = (uint64_t)su < L.P ? (uint64_t)su : L.P;
  { const uint64_t x = (uint64_t)(int64_t)(int32_t)(c.start_unitig + c.nb_unitigs); L.pe = x < L.P ? x : L.P; }
  const uint32_t skip = (uint32_t)(A.k - 1);
  uint64_t name = 0, seq = 0;
  int32_t sr_len = 0;
  bool bad = false;
  auto entry = [&](uint64_t i, uint32_t e) {
    const uint32_t id = e >> 1;
    name += ndigits(id) + 1;
    if((int64_t)i >= su && (int64_t)i < se) sr_len += ulen_of(g, id);
    if(A.useq && i >= L.pb && i < L.pe) {
      if(id >= A.nu) { bad = true; return; }
      const uint64_t sl = A.uoff[id + 1] - A.uoff[id], sk = i == L.pb ? 0 : skip;
      if(sk < sl) seq += sl - sk;
    }
  };
  L.first = walk_path(g, L.b, c.end_node, L.P, entry);
  for(uint64_t i = 0; i < L.first; ++i) entry(i, 0);
  L.name_len = (uint32_t)(name + (L.P ? L.P - 1 : 0));
  sr_len -= (c.nb_unitigs - 1) * (A.k - 1);
  L.sr_len = sr_len;
  L.seq_len = seq;
  L.bad_unitig = bad;
  L.qe_out = (uint64_t)(int64_t)(sr_len + c.end_offset) - ((uint64_t)g.c.ql[L.erow] - (uint64_t)(int64_t)g.c.qe[L.erow]);
  char buf[3 * mrfmt::kFixedMax + 5 * 24];
  L.num_len = (uint32_t)write_numbers(A, L, buf);
  L.sr_digits = (uint32_t)(sr_len < 0 ? 1 + ndigits((uint64_t)0 - (uint64_t)(int64_t)sr_len) : ndigits((uint64_t)sr_len));
  L.len = (uint32_t)(L.hdr + L.num_len + L.name_len + 1 + L.sr_digits + (A.useq ? 1 + L.seq_len : 0) + 1);
}

__global__ void measure_lines_kernel(rec_args A, uint64_t Sc) {
  const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if(l >= Sc) return;
  if(l >= *A.n_lines) { A.line_len[l] = 0; return; }      // (the grid covers the rows; the scan runs over all of them)
  line_t L;
  layout_line(A, l, L);
  if(L.bad_unitig) record_error(A, L.r, kErrUnitig);
  A.line_len[l] = L.len;
  A.line_inf[l] = line_info{ L.pb, L.pe, L.first, L.qe_out, L.hdr, L.num_len, L.name_len, L.sr_len };
}

// the parts of a line's layout that are read from its candidate (layout_line computes the rest)
__device__ __forceinline__ void line_rows(const rec_args& A, uint64_t l, line_t& L) {
  const graph_args& g = A.g;
  L.r = A.line_read[l];
  L.b = g.read_coords[L.r];
  L.c = A.cand + L.b + A.line_node[l];
  L.erow = L.b + L.c->end_node; L.srow = L.b + L.c->start_node;
  L.P = (uint64_t)(g.lunitigs[L.erow] > 0 ? g.lunitigs[L.erow] : 0);
}

__global__ void emit_lines_kernel(rec_args A, uint64_t nlines) {
  const uint64_t l = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if(l >= nlines) return;
  const int lane = (int)lane_id();
  const graph_args& g = A.g;
  line_t L;
  line_rows(A, l, L);
  { const line_info I = A.line_inf[l];
    L.pb = I.pb; L.pe = I.pe; L.first = I.first; L.qe_out = I.qe_out; L.hdr = I.hdr; L.num_len = I.num_len;
    L.name_len = I.name_len; L.sr_len = I.sr_len; }
  char* w = A.text + A.line_off[l];
  char* const end = A.text + (l + 1 < nlines ? A.line_off[l + 1] : A.text_size);
  if(lane == 0) {
    if(L.hdr) {
      *w++ = '>';
      const char* nm = A.names + A.name_off[L.r];
      for(uint32_t i = 0; i + 2 < L.hdr; ++i) *w++ = nm[i];
      *w++ = '\n';
    }
    w += write_numbers(A, L, w);
    // the path's name from its back: "<id><F|R>" joined by '_'
    char* q = w + L.name_len;
    auto put = [&](uint64_t i, uint32_t e) {
      *--q = (e & 1) ? 'R' : 'F';
      uint32_t id = e >> 1;
      do { *--q = (char)('0' + id % 10); id /= 10; } while(id);
      if(i) *--q = '_';
    };
    walk_path(g, L.b, L.c->end_node, L.P, put);
    for(uint64_t i = L.first; i-- > 0;) put(i, 0);
    w += L.name_len;
    *w++ = ' ';
    w += mrfmt::fmt_int(w, L.sr_len);
    if(A.useq) *w++ = ' ';
    end[-1] = '\n';
  }
  if(!A.useq) return;
  // super_read_name::print_sequence (super_read_name.cc:123-132): the pieces from the back, all lanes copying
  char* q = end - 1;
  const uint32_t skip = (uint32_t)(A.k - 1);
  auto piece = [&](uint64_t i, uint32_t e) {
    if(i < L.pb || i >= L.pe) return;
    const uint32_t id = e >> 1;
    const uint64_t o = A.uoff[id], sl = A.uoff[id + 1] - o, sk = i == L.pb ? 0 : skip;
    if(sk >= sl) return;
    const uint64_t n = sl - sk;
    q -= n;
    const char* src = A.useq + o;
    if(e & 1) for(uint64_t j = lane; j < n; j += 32) q[j] = mrfmt::revcomp_base((unsigned char)src[sl - 1 - sk - j]);
    else      for(uint64_t j = lane; j < n; j += 32) q[j] = src[sk + j];
  };
  walk_path(g, L.b, L.c->end_node, L.P, piece);
  for(uint64_t i = L.first; i-- > 0;) piece(i, 0);
}

} // namespace

// read names, through a page-locked staging buffer (the copy then needs no wait for the caller's arrays; the buffer is
// free again because every call that uses it ends with the stream drained)
int upload_read_names(mr_context* ctx, mr_workspace& ws, const char* names, const uint64_t* name_off, uint32_t nreads,
                      const uint64_t** d_off, const char** d_names) {
  const uint64_t name_bytes = name_off[nreads] - name_off[0], off_bytes = ((uint64_t)nreads + 1) * 8;
  MR_TRY(ws.rec_names.ensure(ctx, name_bytes + off_bytes + 64));
  if(ws.rec_names_host.cap < name_bytes + off_bytes + 64) MR_TRY(ws.rec_names_host.ensure(ctx, (name_bytes + off_bytes) * 5 / 4 + 4096));
  uint64_t* h_off = ws.rec_names_host.as<uint64_t>();
  for(uint32_t r = 0; r <= nreads; ++r) h_off[r] = name_off[r] - name_off[0];
  if(name_bytes) memcpy((char*)h_off + off_bytes, names + name_off[0], name_bytes);
  char* q = ws.rec_names.as<char>();
  MR_CUDA(ctx, cudaMemcpyAsync(q, h_off, off_bytes + name_bytes, cudaMemcpyHostToDevice, ctx->stream));
  *d_off = (const uint64_t*)q; *d_names = q + off_bytes;
  return MR_OK;
}

int take_text_slab(mr_context* ctx, mr_workspace& ws, mr_text* t, uint64_t bytes) {
  t->size = bytes;
  {
    std::lock_guard<std::mutex> lock(ws.pool_mutex);
    if(!ws.text_pool.empty()) {                     // the largest slab: the least likely to need regrowing
      size_t best = 0;
      for(size_t i = 1; i < ws.text_pool.size(); ++i) if(ws.text_pool[i]->cap > ws.text_pool[best]->cap) best = i;
      t->host = ws.text_pool[best];
      ws.text_pool.erase(ws.text_pool.begin() + best);
    }
  }
  if(!t->host) t->host = new pinned_buf;
  // a quarter more than this batch needs: batches differ in size, and a slab that is regrown costs a cudaFreeHost (which
  // waits for the device) and a cudaMallocHost of hundreds of megabytes
  if(t->host->cap < bytes + 1 && t->host->ensure(ctx, bytes + bytes / 4 + (1 << 20)) != MR_OK) { delete t->host; t->host = nullptr; return MR_ENOMEM; }
  return MR_OK;
}

extern "C" {

int mr_unitigs_create(mr_context* ctx, const char* seq, const uint64_t* off, uint32_t n, mr_unitigs** out) {
  if(!ctx) return MR_EINVAL;
  if(!seq || !off || !out) return ctx->fail(MR_EINVAL, "mr_unitigs_create: null argument");
  *out = nullptr;
  for(uint32_t i = 0; i < n; ++i)
    if(off[i + 1] < off[i]) return ctx->fail(MR_EINVAL, "mr_unitigs_create: offsets must be non-decreasing");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  std::unique_ptr<mr_unitigs> u(new mr_unitigs);
  u->device = ctx->device; u->n = n;
  const uint64_t bytes = off[n] - off[0];
  MR_TRY(u->seq.ensure(ctx, bytes + 1)); MR_TRY(u->off.ensure(ctx, ((size_t)n + 1) * 8));
  std::vector<uint64_t> rel(off, off + n + 1);
  for(auto& x : rel) x -= off[0];
  if(bytes) MR_CUDA(ctx, cudaMemcpy(u->seq.p, seq + off[0], bytes, cudaMemcpyHostToDevice));
  MR_CUDA(ctx, cudaMemcpy(u->off.p, rel.data(), rel.size() * 8, cudaMemcpyHostToDevice));
  *out = u.release();
  return MR_OK;
}

void mr_unitigs_destroy(mr_unitigs* u) {
  if(!u) return;
  cudaSetDevice(u->device);
  delete u;
}

int mr_records(mr_context* ctx, const mr_result* res, const mr_records_params* p, const mr_unitigs* u,
               const char* names, const uint64_t* name_off, mr_text** out) {
  if(!ctx) return MR_EINVAL;
  if(!res || !p || !names || !name_off || !out) return ctx->fail(MR_EINVAL, "mr_records: null argument");
  *out = nullptr;
  mr_workspace* wsp = ctx->ws;
  if(res->ctx != ctx || !wsp || res->stamp == 0 || res->stamp != wsp->graph_stamp)
    return ctx->fail(MR_EINVAL, "mr_records: the result is not the latest result of this context with an overlap graph");
  if(u && u->device != ctx->device) return ctx->fail(MR_EINVAL, "mr_records: the unitig sequences live on another device");
  if(p->tiling < 0 || p->tiling > 3) return ctx->fail(MR_EINVAL, "mr_records: tiling must be 0 (none), 1 (greedy), 2 (maximal) or 3 (weighted)");
  if(p->unitigs_k == 0) return ctx->fail(MR_EINVAL, "mr_records: -k must be positive");
  MR_CUDA(ctx, cudaSetDevice(ctx->device));
  mr_workspace& ws = *wsp;
  cudaStream_t st = ctx->stream;
  const uint32_t nreads = res->view.nreads;
  const uint64_t S = ws.last_rows, Sc = std::max<uint64_t>(S, 1);
  std::unique_ptr<mr_text> t(new mr_text);
  t->ctx = ctx;
  if(nreads == 0) { *out = t.release(); return MR_OK; }

  rec_args A;
  memset(&A, 0, sizeof A);
  A.g = ws.last_graph;
  A.nreads = nreads;
  A.k = (int32_t)p->unitigs_k;
  A.overlap_play = p->overlap_play; A.density = p->density; A.min_length = p->min_length;
  A.tiling = p->tiling; A.trim = p->trim != 0; A.big_rows = big_rows_threshold();
  // scratch: per row a candidate, 7 ints, a double, two spans and a tiling entry; per read the line counts
  MR_TRY(ws.rec_cand.ensure(ctx, Sc * sizeof(cand_t)));
  MR_TRY(ws.rec_i32.ensure(ctx, Sc * 4 * 9 + 64));
  MR_TRY(ws.rec_f64.ensure(ctx, Sc * (8 + 2 * 16)));
  MR_TRY(ws.rec_info.ensure(ctx, Sc * sizeof(tinfo_t)));
  MR_TRY(ws.rec_lines.ensure(ctx, Sc * 8 + ((size_t)nreads + 2) * 12 + 64));
  MR_TRY(ws.rec_linf.ensure(ctx, Sc * sizeof(line_info)));
  A.line_inf = ws.rec_linf.as<line_info>();
  A.cand = ws.rec_cand.as<cand_t>();
  { int32_t* q = ws.rec_i32.as<int32_t>(); A.comp_slot = q; A.comp_best = q + Sc; A.mrs = q + 2 * Sc; A.sort_t = q + 3 * Sc;
    A.tiled = q + 4 * Sc; A.order = q + 5 * Sc; A.line_node = q + 6 * Sc; A.line_read = (uint32_t*)(q + 7 * Sc); A.line_len = (uint32_t*)(q + 8 * Sc);
    A.err = (unsigned long long*)(((uintptr_t)(q + 9 * Sc) + 15) & ~(uintptr_t)15); }
  { char* q = ws.rec_f64.as<char>(); A.cov = (double2*)q; A.placed = (double2*)(q + Sc * 16); A.weight = (double*)(q + Sc * 32); }
  A.info = ws.rec_info.as<tinfo_t>();
  { char* q = ws.rec_lines.as<char>(); A.line_off = (uint64_t*)q; A.line_base = (uint64_t*)(q + Sc * 8);
    A.nlines = (uint32_t*)(q + Sc * 8 + ((size_t)nreads + 2) * 8); }
  uint64_t* d_tot = (uint64_t*)A.err + 1;        // [0] lines, [1] bytes
  A.n_lines = d_tot;
  MR_TRY(upload_read_names(ctx, ws, names, name_off, nreads, &A.name_off, &A.names));
  if(u) { A.useq = u->seq.as<char>(); A.uoff = u->off.as<uint64_t>(); A.nu = u->n; }
  MR_CUDA(ctx, cudaMemsetAsync(A.err, 0xff, 8, st));
  MR_CUDA(ctx, cudaMemsetAsync(d_tot, 0, 16, st));

  uint64_t h[3] = { ~0ULL, 0, 0 };
  if(nreads) {
    plan_small_kernel<<<div_up(nreads, 128), 128, 0, st>>>(A);
    MR_LAUNCHED(ctx);
    if(ws.last_max_rows > A.big_rows) {
      plan_big_kernel<<<div_up((uint64_t)nreads * 32, 256), 256, 0, st>>>(A);
      MR_LAUNCHED(ctx);
    }
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ A.nlines }, nreads, A.line_base, ws.scan_scratch, d_tot)));
    expand_lines_kernel<<<div_up(nreads, 128), 128, 0, st>>>(A);
    MR_LAUNCHED(ctx);
    measure_lines_kernel<<<div_up(Sc, 128), 128, 0, st>>>(A, Sc);
    MR_LAUNCHED(ctx);
    MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ A.line_len }, Sc, A.line_off, ws.scan_scratch, d_tot + 1)));
    MR_CUDA(ctx, cudaMemcpyAsync(h, A.err, 24, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
  }
  if(h[0] != ~0ULL)
    return ctx->fail(MR_EINVAL, (h[0] & 1) ? "unitig id of a super-read name is not in the -u file"
                                           : "component root outside the read's rows");
  const uint64_t nlines = h[1], bytes = h[2];
  MR_TRY(take_text_slab(ctx, ws, t.get(), bytes));
  if(nlines) {
    MR_TRY(ws.rec_text.ensure(ctx, bytes + 1));
    A.text = ws.rec_text.as<char>();
    A.text_size = bytes;
    emit_lines_kernel<<<div_up(nlines * 32, 256), 256, 0, st>>>(A, nlines);
    MR_LAUNCHED(ctx);
    MR_CUDA(ctx, cudaMemcpyAsync(t->host->p, A.text, bytes, cudaMemcpyDeviceToHost, st));
    MR_CUDA(ctx, ctx->wait(st));
  }
  *out = t.release();
  return MR_OK;
}

int mr_text_get(const mr_text* t, const char** bytes, uint64_t* size) {
  if(!t || !bytes || !size) return MR_EINVAL;
  *bytes = t->size ? t->host->as<char>() : "";
  *size = t->size;
  return MR_OK;
}

void mr_text_free(mr_text* t) {
  if(!t) return;
  if(t->host) {
    bool kept = false;
    mr_workspace* ws = t->ctx->ws;
    if(ws) {
      std::lock_guard<std::mutex> lock(ws->pool_mutex);
      if(ws->text_pool.size() < 4) { ws->text_pool.push_back(t->host); kept = true; }
    }
    if(!kept) { cudaSetDevice(t->ctx->device); delete t->host; }
  }
  delete t;
}

} // extern "C"

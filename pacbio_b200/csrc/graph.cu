// Overlap graph between the super-reads aligned to one read: nodes ordered by implied start,
// O(n^2) edge test (position overlap vs unitig-path dovetail overlap), longest-path DP and
// union-find components.  One warp per read (graph_kernel) or, for a read with many rows, one CTA
// (graph_big_kernel); the outer node loop is sequential as in the reference, the inner loop over
// candidate successors runs 32 (256) wide with a ballot for the reference's `break`.  Replaces overlap_graph::thread::reset + overlap_graph::traverse
// (overlap_graph.hpp:24-34,177-196, overlap_graph.cc:7-59, union_find.cc:6-24,
// super_read_name.cc:49-72).
#include "align.cuh"

namespace {

struct path_ref {
  const uint32_t* ids; uint32_t n; bool bwd;
  __device__ uint32_t at(uint32_t t) const { return bwd ? (ids[n - 1 - t] ^ 1u) : ids[t]; }
};

__device__ __forceinline__ path_ref row_path(const graph_args& A, uint64_t row) {
  path_ref p;
  if(!A.unitig_off) { p.ids = nullptr; p.n = 0; p.bwd = false; return p; }
  const uint32_t sr = A.c.sr[row];
  const uint64_t u0 = A.unitig_off[sr];
  p.ids = A.unitig_ids + u0;
  p.n   = (uint32_t)(A.unitig_off[sr + 1] - u0);
  p.bwd = A.c.use_bwd[row] != 0;
  return p;
}

// largest t such that the last t unitigs of l equal the first t of r (super_read_name.cc:49-72)
__device__ int dovetail(const path_ref& l, const path_ref& r) {
  if(l.n < 2 || r.n < 2) return 0;
  int32_t first = (int32_t)l.n - (int32_t)r.n + 1;
  if(first < 1) first = 1;
  const uint32_t r0 = r.at(0);
  for(uint32_t i = (uint32_t)first; i < l.n; ++i) {
    if(l.at(i) != r0) continue;
    uint32_t j = i + 1;
    while(j < l.n && l.at(j) == r.at(j - i)) ++j;
    if(j == l.n) return (int)(l.n - i);
  }
  return 0;
}

__device__ bool same_path(const path_ref& a, const path_ref& b) {
  if(a.n != b.n) return false;
  for(uint32_t t = 0; t < a.n; ++t) if(a.at(t) != b.at(t)) return false;
  return true;
}

__device__ int uf_find(int32_t* parent, int s) {
  int r = s;
  while(parent[r] != r) r = parent[r];
  while(parent[s] != r) { const int nx = parent[s]; parent[s] = r; s = nx; }
  return r;
}

__global__ void __launch_bounds__(128) graph_kernel(graph_args A) {
  __shared__ int32_t edge_j[4][32];
  const unsigned lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if(r >= A.nreads) return;
  const uint64_t b = A.read_coords[r];
  const int n = (int)(A.read_coords[r + 1] - b);
  if(n == 0 || n > A.warp_max_rows) return;           // many rows: graph_big_kernel
  const double rl = (double)A.read_len[r];
  const double K = (double)A.unitigs_k;
  int32_t* parent = A.component + b;
  int32_t* rank   = A.uf_rank + b;
  int32_t* order  = A.order + b;
  double*  imp_s  = A.imp_s + b;
  double*  imp_e  = A.imp_e + b;

  // node_info::reset (overlap_graph.hpp:24-34)
  for(int i = lane; i < n; i += 32) {
    const uint64_t row = b + i;
    const double st = A.c.stretch[row], of = A.c.offset[row];
    imp_s[i] = st + of;
    const double t = st * (double)A.c.ql[row];
    imp_e[i] = t + of;
    A.start_node[row] = 1; A.end_node[row] = 1;
    parent[i] = i; rank[i] = 0;
    A.lstart[row] = -1; A.lprev[row] = -1;
    A.lpath[row] = A.bases ? (int32_t)A.c.sr_cover[row] : A.c.nb_mers[row];
    A.lunitigs[row] = (int32_t)row_path(A, row).n;
  }
  __syncwarp();
  // node order by (imp_s, imp_e); exact ties keep row order (the reference's std::sort is unstable there)
  for(int i = lane; i < n; i += 32) {
    const double s = imp_s[i], e = imp_e[i];
    int rk = 0;
    for(int j = 0; j < n; ++j) {
      const double sj = imp_s[j], ej = imp_e[j];
      rk += (sj < s || (sj == s && ej < e)) || (sj == s && ej == e && j < i);
    }
    order[rk] = i;
  }
  __syncwarp();

  for(int a = 0; a < n; ++a) {
    const int ii = order[a];
    const uint64_t row_i = b + ii;
    const double ie_i = imp_e[ii];
    if(ie_i >= rl) continue;                         // hanging off the 3' end of the read
    const path_ref pi = row_path(A, row_i);
    const double err_i = A.c.avg_err[row_i];
    const int lpath_i = A.lpath[row_i], lstart_i = A.lstart[row_i], lunitigs_i = A.lunitigs[row_i];
    const double start_s_i = imp_s[lstart_i == -1 ? ii : lstart_i];
    bool any_edge = false;
    for(int b0 = a + 1; b0 < n; b0 += 32) {
      const int bb = b0 + (int)lane;
      const bool in = bb < n;
      const int jj = in ? order[bb] : 0;
      const uint64_t row_j = b + jj;
      const double is_j = imp_s[jj], ie_j = imp_e[jj];
      const bool skip = !in || is_j <= 1 || ie_i > ie_j + 31;
      const double position_len = ie_i - is_j;
      const double error1 = err_i + A.c.avg_err[row_j];
      const double error  = A.errors * error1;
      const double ppl = position_len * A.overlap_play;
      const bool brk = !skip && (ppl + error < K);
      const unsigned ball = __ballot_sync(MR_FULL_MASK, brk);
      const unsigned limit = ball ? (unsigned)(__ffs(ball) - 1) : 32u;
      bool edge = false;
      int nb_u = 0, common = 0;
      path_ref pj; pj.ids = nullptr; pj.n = 0; pj.bwd = false;
      if(!skip && lane < limit) {
        pj = row_path(A, row_j);
        nb_u = dovetail(pi, pj);
        if(nb_u && !same_path(pi, pj)) {
          int u_overlap_len = 0;
          const uint32_t ilen = A.c.info_len[row_j];
          const int32_t* info = (A.bases ? A.binfo : A.kinfo) + A.c.info_off[row_j];
          for(int u = 0; u < nb_u; ++u) {
            u_overlap_len += A.unitig_len[pj.at(u) >> 1];
            if((uint32_t)(2 * u) < ilen) common += info[2 * u];
            if(u > 0 && (uint32_t)(2 * u - 1) < ilen) common -= info[2 * u - 1];
          }
          u_overlap_len -= (nb_u - 1) * ((int)A.unitigs_k - 1);
          const double t1 = A.overlap_play * position_len;
          const double t2 = A.overlap_play * ((double)u_overlap_len + error);
          edge = !((double)u_overlap_len > t1 + error || position_len > t2);
        }
      }
      const unsigned eb = __ballot_sync(MR_FULL_MASK, edge);
      if(eb) {
        any_edge = true;
        if(edge) {
          A.start_node[row_j] = 0;
          const int nlpath = lpath_i + (A.bases ? (int)A.c.sr_cover[row_j] : A.c.nb_mers[row_j]) - common;
          const int lpath_j = A.lpath[row_j], lstart_j = A.lstart[row_j];
          const double start_s_j = imp_s[lstart_j == -1 ? jj : lstart_j];
          if(nlpath > lpath_j || (nlpath == lpath_j && (lstart_j == -1 || start_s_i > start_s_j))) {
            A.lpath[row_j]    = nlpath;
            A.lstart[row_j]   = lstart_i == -1 ? ii : lstart_i;
            A.lprev[row_j]    = ii;
            A.lunitigs[row_j] = lunitigs_i + (int)pj.n - nb_u;
          }
        }
        // components: unions in successor order, exactly as the sequential loop would do them
        edge_j[wib][lane] = jj;
        __syncwarp();
        if(lane == 0) {
          unsigned m = eb;
          while(m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const int r1 = uf_find(parent, ii), r2 = uf_find(parent, edge_j[wib][src]);
            if(rank[r1] > rank[r2]) parent[r2] = r1;
            else if(rank[r1] < rank[r2]) parent[r1] = r2;
            else if(r1 != r2) { parent[r2] = r1; ++rank[r1]; }
          }
        }
        __syncwarp();
      }
      if(ball) break;
    }
    if(any_edge && lane == 0) A.end_node[row_i] = 0;
    __syncwarp();
  }

  // component root of every node (union_find::set::root)
  for(int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + (int)lane;
    int root = 0;
    if(i < n) { root = i; while(parent[root] != root) root = parent[root]; }
    __syncwarp();
    if(i < n) parent[i] = root;
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// Reads with many rows (repeats: hundreds to thousands of super-reads stacked on one read).  The
// reference's loop (overlap_graph.cc:7-59) does two different things for a pair (i, j): a TEST that
// depends on the two nodes alone (positions, unitig-path dovetail, matched mers they share) and an
// UPDATE of the longest-path and union-find state, which is sequential.  Here the tests of all
// pairs of a read -- 35 M per 32-Mbase batch of human-shaped reads, of which 5 M are edges -- run
// first, one warp per node, in parallel over the whole batch; only the surviving edges reach the
// sequential part, which one CTA per read runs out of shared memory.
//   graph_big_prepare_kernel  node_info::reset + node order (overlap_graph.hpp:24-34,177-196)
//   graph_edges_kernel<false> counts the out-edges of every node; <true> writes them, compacted, in
//                             successor order (the slices come from an exclusive scan of the counts)
//   graph_path_kernel         warp 0: components (union_find.cc:6-24) in edge order; warp 1: longest path
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) graph_big_prepare_kernel(graph_args A, int sort_cap) {
  const int tid = (int)threadIdx.x;
  const uint32_t r = blockIdx.x;
  if(r >= A.nreads) return;
  const uint64_t b = A.read_coords[r];
  const int n = (int)(A.read_coords[r + 1] - b);
  if(n <= A.warp_max_rows) return;
  int32_t* order  = A.order + b;
  double*  imp_s  = A.imp_s + b;
  double*  imp_e  = A.imp_e + b;
  // the values a successor scan needs, in node ORDER: consecutive candidates are consecutive in memory
  double*  ord_s   = A.ord_s + b;
  double*  ord_e   = A.ord_e + b;
  double*  ord_err = A.ord_err + b;
  ulonglong2* ord_path = A.ord_path + b;

  for(int i = tid; i < n; i += 256) {
    const uint64_t row = b + i;
    const double st = A.c.stretch[row], of = A.c.offset[row];
    imp_s[i] = st + of;
    const double t = st * (double)A.c.ql[row];
    imp_e[i] = t + of;
    A.start_node[row] = 1; A.end_node[row] = 1;
  }
  __syncthreads();
  // node order by (imp_s, imp_e), exact ties by row (the reference's std::sort is unstable there)
  auto place = [&](int rk, int i) {
    const uint64_t row = b + i;
    order[rk] = i;
    ord_s[rk] = imp_s[i]; ord_e[rk] = imp_e[i]; ord_err[rk] = A.c.avg_err[row];
    const uint32_t sr = A.c.sr[row];
    const uint64_t u0 = A.unitig_off ? A.unitig_off[sr] : 0;
    const uint32_t un = A.unitig_off ? (uint32_t)(A.unitig_off[sr + 1] - u0) : 0u;
    ord_path[rk] = make_ulonglong2(u0, (uint64_t)un | ((uint64_t)(A.c.use_bwd[row] != 0) << 32));
  };
  if(n <= sort_cap) {
    // bitonic sort of the node indices with their keys in shared memory
    extern __shared__ __align__(16) unsigned char dyn[];
    double* ks = (double*)dyn;
    double* ke = ks + sort_cap;
    uint32_t* idx = (uint32_t*)(ke + sort_cap);
    int m = 1;
    while(m < n) m <<= 1;
    for(int i = tid; i < m; i += 256) {
      if(i < n) { ks[i] = imp_s[i]; ke[i] = imp_e[i]; idx[i] = (uint32_t)i; }
      else idx[i] = prim::kPad;
    }
    __syncthreads();
    prim::bitonic_sort_idx(idx, m, [&](uint32_t x, uint32_t y) {
      const double sx = ks[x], sy = ks[y];
      if(sx != sy) return sx < sy;
      const double ex = ke[x], ey = ke[y];
      return ex != ey ? ex < ey : x < y;
    });
    for(int rk = tid; rk < n; rk += 256) place(rk, (int)idx[rk]);
    return;
  }
  // larger reads: by counting, 256 nodes at a time against all nodes, which pass through shared memory in tiles
  __shared__ double2 tile[256];
  for(int i0 = 0; i0 < n; i0 += 256) {
    const int i = i0 + tid;
    const bool mine = i < n;
    const double s = mine ? imp_s[i] : 0.0, e = mine ? imp_e[i] : 0.0;
    int rk = 0;
    for(int j0 = 0; j0 < n; j0 += 256) {
      __syncthreads();
      if(j0 + tid < n) tile[tid] = make_double2(imp_s[j0 + tid], imp_e[j0 + tid]);
      __syncthreads();
      const int mm = min(256, n - j0);
#pragma unroll 4
      for(int j = 0; j < mm; ++j) {
        const double2 o = tile[j];
        rk += (o.x < s || (o.x == s && o.y < e)) || (o.x == s && o.y == e && j0 + j < i);
      }
    }
    if(mine) place(rk, i);
  }
}

// One warp per node (a row of a read with many rows; the warps of all other rows leave at once).
// Lane l tests the node's l-th, (32 + l)-th, ... successor in node order; the reference's `break` is the
// first flagged lane of a round.  An edge is {successor's order position, weight - common, unitigs added}.
template<bool kWrite>
__global__ void __launch_bounds__(256) graph_edges_kernel(graph_args A, uint64_t S) {
  const unsigned lane = threadIdx.x & 31;
  const uint64_t g = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if(g >= S) return;
  const uint32_t r = A.c.read[g];
  const uint64_t b = A.read_coords[r];
  const int n = (int)(A.read_coords[r + 1] - b);
  if(n <= A.warp_max_rows) { if(!kWrite && lane == 0) A.edge_cnt[g] = 0; return; }
  const int a = (int)(g - b);
  const double* ord_s = A.ord_s + b;
  const double* ord_e = A.ord_e + b;
  const double* ord_err = A.ord_err + b;
  const ulonglong2* ord_path = A.ord_path + b;
  const int32_t* order = A.order + b;
  const double rl = (double)A.read_len[r];
  const double K = (double)A.unitigs_k;
  const double ie_i = ord_e[a];
  uint32_t count = 0;
  if(ie_i < rl) {                                        // else: hanging off the 3' end of the read, no successors
    const double err_i = ord_err[a];
    const ulonglong2 dpi = ord_path[a];
    path_ref pi; pi.ids = A.unitig_ids + dpi.x; pi.n = (uint32_t)dpi.y; pi.bwd = (dpi.y >> 32) != 0;
    int4* out = kWrite ? A.edges + A.edge_off[g] : nullptr;
    for(int b0 = a + 1; b0 < n; b0 += 32) {
      const int bb = b0 + (int)lane;
      const bool in = bb < n;
      const double is_j = in ? ord_s[bb] : 0.0, ie_j = in ? ord_e[bb] : 0.0;
      const bool skip = !in || is_j <= 1 || ie_i > ie_j + 31;
      const double position_len = ie_i - is_j;
      const double error1 = err_i + (in ? ord_err[bb] : 0.0);
      const double error  = A.errors * error1;
      const double ppl = position_len * A.overlap_play;
      const bool brk = !skip && (ppl + error < K);
      const unsigned ball = __ballot_sync(MR_FULL_MASK, brk);
      const unsigned limit = ball ? (unsigned)(__ffs(ball) - 1) : 32u;
      bool edge = false;
      int delta = 0, add = 0, jj = 0;
      if(!skip && lane < limit) {
        const ulonglong2 dpj = ord_path[bb];
        path_ref pj; pj.ids = A.unitig_ids + dpj.x; pj.n = (uint32_t)dpj.y; pj.bwd = (dpj.y >> 32) != 0;
        const int nb_u = dovetail(pi, pj);
        if(nb_u && !same_path(pi, pj)) {
          jj = order[bb];
          const uint64_t row_j = b + jj;
          int u_overlap_len = 0, common = 0;
          const uint32_t ilen = A.c.info_len[row_j];
          const int32_t* info = (A.bases ? A.binfo : A.kinfo) + A.c.info_off[row_j];
          for(int u = 0; u < nb_u; ++u) {
            u_overlap_len += A.unitig_len[pj.at(u) >> 1];
            if((uint32_t)(2 * u) < ilen) common += info[2 * u];
            if(u > 0 && (uint32_t)(2 * u - 1) < ilen) common -= info[2 * u - 1];
          }
          u_overlap_len -= (nb_u - 1) * ((int)A.unitigs_k - 1);
          const double t1 = A.overlap_play * position_len;
          const double t2 = A.overlap_play * ((double)u_overlap_len + error);
          edge = !((double)u_overlap_len > t1 + error || position_len > t2);
          if(edge && kWrite) {
            delta = (A.bases ? (int)A.c.sr_cover[row_j] : A.c.nb_mers[row_j]) - common;
            add = (int)pj.n - nb_u;
          }
        }
      }
      const unsigned eb = __ballot_sync(MR_FULL_MASK, edge);
      if(kWrite && edge) {
        out[count + __popc(eb & lanemask_lt())] = make_int4(bb, delta, add, 0);
        A.start_node[b + jj] = 0;
      }
      count += __popc(eb);
      if(ball) break;
    }
  }
  if(lane == 0) {
    if(!kWrite) A.edge_cnt[g] = count;
    else if(count) A.end_node[b + order[a]] = 0;
  }
}

// Sequential part of a read with many rows, over its edges only.  64 threads: warp 0 does the unions in
// the reference's order (node by node, successors ascending), warp 1 the longest-path updates; they
// share nothing but the read-only edge list.  State is indexed by ORDER POSITION and lives in shared
// memory (33 bytes per node) when the read has at most `cap` rows, else in the global scratch slices.
//   unions: lanes find the roots of 32 edges at once; edges whose ends already share a root are
//           no-ops (most of them in a dense stack), the first one that does not is performed and the
//           roots held by the other lanes are patched -- so a chunk costs one round of finds plus one
//           short step per EFFECTIVE union, and the order of effective unions, hence every rank and
//           root, is the sequential one.
//   longest path: the out-edges of one node go to distinct successors, so they update in parallel.
struct path_scratch { int32_t* i32; double* f64; uint8_t* u8; };    // global fallback: 6 x int32, 1 x double, 1 x uint8 per row
__global__ void __launch_bounds__(64) graph_path_kernel(graph_args A, int cap, int cap_alloc, path_scratch G) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t r = blockIdx.x;
  if(r >= A.nreads) return;
  const uint64_t b = A.read_coords[r];
  const int n = (int)(A.read_coords[r + 1] - b);
  if(n <= A.warp_max_rows) return;
  double* start_s; int32_t *lpath, *lstart, *lprev, *lunitigs, *parent, *cnt; uint8_t* rank;
  if(n <= cap) {
    unsigned char* p = smem_raw;
    start_s = (double*)p;   p += (size_t)cap_alloc * 8;
    lpath = (int32_t*)p;    p += (size_t)cap_alloc * 4;
    lstart = (int32_t*)p;   p += (size_t)cap_alloc * 4;
    lprev = (int32_t*)p;    p += (size_t)cap_alloc * 4;
    lunitigs = (int32_t*)p; p += (size_t)cap_alloc * 4;
    parent = (int32_t*)p;   p += (size_t)cap_alloc * 4;
    cnt = (int32_t*)p;      p += (size_t)cap_alloc * 4;
    rank = (uint8_t*)p;
  } else {
    const uint64_t S = A.read_coords[A.nreads];
    start_s = G.f64 + b;
    lpath = G.i32 + b; lstart = G.i32 + S + b; lprev = G.i32 + 2 * S + b; lunitigs = G.i32 + 3 * S + b;
    parent = G.i32 + 4 * S + b; cnt = G.i32 + 5 * S + b;
    rank = G.u8 + b;
  }
  const int32_t* order = A.order + b;
  const double*  ord_s = A.ord_s + b;
  for(int p = (int)threadIdx.x; p < n; p += 64) {
    const uint64_t row = b + order[p];
    start_s[p] = ord_s[p];
    lpath[p] = A.bases ? (int32_t)A.c.sr_cover[row] : A.c.nb_mers[row];
    lstart[p] = -1; lprev[p] = -1;
    lunitigs[p] = (int32_t)(uint32_t)A.ord_path[b + p].y;
    parent[p] = p; rank[p] = 0;
    cnt[p] = (int32_t)A.edge_cnt[b + p];
  }
  __syncthreads();
  const int4* edges = A.edges + A.edge_off[b];
  if(warp == 0) {
    // ---- components ---------------------------------------------------------------------------
    uint64_t off = 0;
    for(int a = 0; a < n; ++a) {
      const int c = cnt[a];
      for(int c0 = 0; c0 < c; c0 += 32) {
        const bool have = c0 + (int)lane < c;
        int ri, rj = -1;
        {                                             // find with path compression: every write stores an ancestor
          int x = a, rt = a;
          while(parent[rt] != rt) rt = parent[rt];
          while(parent[x] != rt) { const int nx = parent[x]; parent[x] = rt; x = nx; }
          ri = rt;
        }
        if(have) {
          int x = edges[off + c0 + lane].x, rt = x;
          while(parent[rt] != rt) rt = parent[rt];
          while(parent[x] != rt) { const int nx = parent[x]; parent[x] = rt; x = nx; }
          rj = rt;
        }
        __syncwarp();
        while(true) {
          const unsigned m = __ballot_sync(MR_FULL_MASK, have && ri != rj);
          if(!m) break;
          const int f = __ffs(m) - 1;
          const int r1 = __shfl_sync(MR_FULL_MASK, ri, f), r2 = __shfl_sync(MR_FULL_MASK, rj, f);
          const int k1 = rank[r1], k2 = rank[r2];
          const int win = k1 >= k2 ? r1 : r2, lose = k1 >= k2 ? r2 : r1;
          if(lane == 0) { parent[lose] = win; if(k1 == k2) rank[r1] = (uint8_t)(k1 + 1); }
          if(ri == lose) ri = win;
          if(rj == lose) rj = win;
          __syncwarp();
        }
      }
      off += (uint64_t)c;
    }
    __syncwarp();
    // component root of every node, as a row offset inside the read (union_find::set::root)
    for(int p = (int)lane; p < n; p += 32) {
      int rt = p;
      while(parent[rt] != rt) rt = parent[rt];
      A.component[b + order[p]] = order[rt];
    }
  } else {
    // ---- longest path -----------------------------------------------------------------------
    uint64_t off = 0;
    for(int a = 0; a < n; ++a) {
      const int c = cnt[a];
      if(c == 0) continue;
      const int lpath_i = lpath[a], lstart_i = lstart[a], lun_i = lunitigs[a];
      const double start_s_i = start_s[a];
      for(int q = (int)lane; q < c; q += 32) {
        const int4 e = edges[off + q];
        const int nl = lpath_i + e.y;
        const int lpath_j = lpath[e.x], lstart_j = lstart[e.x];
        if(nl > lpath_j || (nl == lpath_j && (lstart_j == -1 || start_s_i > start_s[e.x]))) {
          lpath[e.x] = nl;
          lstart[e.x] = lstart_i == -1 ? a : lstart_i;
          lprev[e.x] = a;
          lunitigs[e.x] = lun_i + e.z;
          start_s[e.x] = start_s_i;
        }
      }
      off += (uint64_t)c;
      __syncwarp();
    }
    for(int p = (int)lane; p < n; p += 32) {
      const uint64_t row = b + order[p];
      A.lpath[row] = lpath[p];
      A.lstart[row] = lstart[p] == -1 ? -1 : order[lstart[p]];
      A.lprev[row] = lprev[p] == -1 ? -1 : order[lprev[p]];
      A.lunitigs[row] = lunitigs[p];
    }
  }
}

} // namespace

// max_rows: the largest number of rows any read of the batch has (known on the host)
int launch_graph(mr_context* ctx, mr_workspace& ws, graph_args a, uint64_t S, int max_rows) {
  if(a.nreads == 0 || S == 0) return MR_OK;
  cudaStream_t st = ctx->stream;
  graph_kernel<<<div_up((uint64_t)a.nreads * 32, 128), 128, 0, st>>>(a);
  MR_LAUNCHED(ctx);
  if(max_rows <= a.warp_max_rows) return MR_OK;
  // ---- reads with many rows: parallel edge pass, then the sequential part over edges only ----------
  MR_TRY(ws.counters.ensure(ctx, 16 * sizeof(uint64_t)));
  MR_TRY(ws.node_path.ensure(ctx, S * sizeof(ulonglong2)));
  MR_TRY(ws.edge_cnt.ensure(ctx, (S + 1) * sizeof(uint32_t)));
  MR_TRY(ws.edge_off.ensure(ctx, (S + 2) * sizeof(uint64_t)));
  a.ord_path = ws.node_path.as<ulonglong2>(); a.edge_cnt = ws.edge_cnt.as<uint32_t>(); a.edge_off = ws.edge_off.as<uint64_t>();
  a.edges = nullptr;
  {
    // node order: bitonic sort in shared memory (20 bytes per row, rounded up to a power of two) up to 4096 rows
    int sort_cap = 1;
    while(sort_cap < std::min(max_rows, big_sort_rows_limit())) sort_cap <<= 1;
    if(sort_cap > big_sort_rows_limit()) sort_cap >>= 1;
    const size_t smem = (size_t)sort_cap * 20;
    MR_CUDA(ctx, cudaFuncSetAttribute(graph_big_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    graph_big_prepare_kernel<<<a.nreads, 256, smem, st>>>(a, sort_cap);
    MR_LAUNCHED(ctx);
  }
  const unsigned node_blocks = div_up(S * 32, 256);
  graph_edges_kernel<false><<<node_blocks, 256, 0, st>>>(a, S);
  MR_LAUNCHED(ctx);
  MR_CUDA(ctx, cudaMemsetAsync(a.edge_cnt + S, 0, sizeof(uint32_t), st));
  unsigned long long* d_total = ws.counters.as<unsigned long long>() + 13;
  MR_TRY((prim::exclusive_scan<prim::ptr_in_u32, uint64_t>(ctx, prim::ptr_in_u32{ a.edge_cnt }, S + 1, a.edge_off, ws.scan_scratch, (uint64_t*)d_total)));
  uint64_t E = 0;
  MR_CUDA(ctx, cudaMemcpyAsync(&E, d_total, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  MR_CUDA(ctx, cudaStreamSynchronize(st));
  MR_TRY(ws.edges.ensure(ctx, (E + 1) * sizeof(int4)));
  a.edges = ws.edges.as<int4>();
  if(E) {
    graph_edges_kernel<true><<<node_blocks, 256, 0, st>>>(a, S);
    MR_LAUNCHED(ctx);
  }
  // shared memory of the sequential kernel: 33 bytes per row of the largest read, up to what a CTA may have
  const int cap = std::min(max_rows, path_smem_rows_limit());
  const int cap_alloc = (cap + 63) / 64 * 64;
  const size_t smem = (size_t)cap_alloc * 33 + 64;
  path_scratch G = { nullptr, nullptr, nullptr };
  if(max_rows > cap) {                                   // some read does not fit: its state goes to global scratch
    MR_TRY(ws.path_i32.ensure(ctx, S * 6 * sizeof(int32_t))); MR_TRY(ws.path_f64.ensure(ctx, S * sizeof(double)));
    MR_TRY(ws.path_u8.ensure(ctx, S));
    G.i32 = ws.path_i32.as<int32_t>(); G.f64 = ws.path_f64.as<double>(); G.u8 = ws.path_u8.as<uint8_t>();
  }
  MR_CUDA(ctx, cudaFuncSetAttribute(graph_path_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  graph_path_kernel<<<a.nreads, 64, smem, st>>>(a, cap, cap_alloc, G);
  MR_LAUNCHED(ctx);
  return MR_OK;
}

// Shared declarations for the per-batch alignment pipeline (align.cu, graph.cu, result.cu).
#pragma once
#include <algorithm>
#include <cstdlib>
#include "index.cuh"
#include "primitives.cuh"

#include <mutex>

constexpr int      kTile        = 1024;           // read positions per CTA in the seed / expand kernels
constexpr int      kSeedThreads = 256;
constexpr uint32_t kNone        = 0xffffffffu;

// a batch of reads on the device, 2-bit packed + non-ACGT mask (align.cu, load_tile_codes)
struct packed_reads {
  const uint64_t* __restrict__ codes;
  const uint64_t* __restrict__ nmask;
  int tma;                            // both arrays are 16-byte aligned: tiles are staged with bulk copies
};

// Final per-coords arrays on the device (structure of arrays, rows sorted per read).
struct coords_soa {
  int32_t  *rs, *re, *qs, *qe, *nb_mers;
  uint32_t *pb_cons, *sr_cons, *pb_cover, *sr_cover, *ql, *sr, *read;
  uint8_t  *rn, *use_bwd;
  double   *stretch, *offset, *avg_err;
  uint64_t *info_off;
  uint32_t *info_len;
  uint64_t *chain_pos;     // start of the group's slice in the sorted hit arrays
};

// scratch of the fine pass
struct fine_buffers {
  dev_buf wkey0, wkey1, wrow0, wrow1, wbegin, wend, gread, gsr, giter, table_off, row_cnt, group_start;
  prim::sort_scratch sort;
};

// a batch of reads already copied (or on its way) to the device, see mr_stage_batch
struct mr_staged {
  mr_context* ctx = nullptr;
  dev_buf bases, read_start;          // bases: characters, or with `packed` the code words followed by the mask words
  bool packed = false;
  std::vector<uint64_t> h_read_start;
  uint32_t nreads = 0;
  cudaEvent_t ready = nullptr;
  ~mr_staged() { if(ready) cudaEventDestroy(ready); }
};

// graph.cu
struct graph_args {
  uint32_t nreads;
  const uint64_t* read_coords;
  const uint32_t* read_len;
  coords_soa c;
  const int32_t *kinfo, *binfo;
  const uint32_t* unitig_ids; const uint64_t* unitig_off; const int32_t* unitig_len;
  uint32_t n_unitigs, unitigs_k;
  double overlap_play, errors;
  int bases;
  int warp_max_rows;       // reads with more rows than this take the edge-list kernels instead of one warp (big_rows_threshold())
  double *ord_s, *ord_e, *ord_err;   // reads with many rows: imp_s, imp_e, avg_err in node order
  ulonglong2* ord_path;              // ... and the node's unitig path: x = offset into unitig_ids, y = length | reversed << 32
  uint32_t*   edge_cnt;              // out-edges of the node at every order position (0 for the rows of other reads)
  uint64_t*   edge_off;              // exclusive scan of edge_cnt: a node's slice of `edges`
  int4*       edges;                 // { successor's order position, weight - common, unitigs added, 0 }
  // outputs / scratch, one entry per row
  uint8_t *start_node, *end_node;
  int32_t *lstart, *lprev, *lpath, *lunitigs, *component, *uf_rank, *order;
  double  *imp_s, *imp_e;
};

// The final rows of a batch where it left them on the device (mr_coords_records reads them there).
struct rows_args {
  uint32_t nreads;
  uint64_t nrows;
  const uint64_t* read_coords;
  const uint32_t* read_len;
  coords_soa c;
  const int32_t *kinfo, *binfo;
};

// Scratch that lives in the context and is reused from batch to batch.
struct mr_workspace {
  dev_buf bases, codes, nmask, read_start, read_len, tile_read, tile_pos, tile_first, tile_cand, tile_tbase;
  dev_buf size, rec, hit_off, thr, counters;
  fine_buffers fine;
  dev_buf path_ids, path_off, path_ulen;               // mr_graph_batch: the caller's unitig paths
  dev_buf key0, key1, pay0, pay1, chainL, group_start, head;
  dev_buf sv_i32, sv_u32, sv_f64, sv_u64, sv_u8;        // survivors, unsorted
  dev_buf fin_i32, fin_u32, fin_f64, fin_u64, fin_u8;   // final rows
  dev_buf read_cnt, read_coords, read_cursor, slot, order, rowkey4, rowkey5;
  dev_buf kinfo, binfo;
  dev_buf node_i32, node_u8, node_f64;
  dev_buf node_path, edge_cnt, edge_off, edges, path_i32, path_f64, path_u8;   // overlap graph of reads with many rows (graph.cu)
  dev_buf tap_lens, tap_cf, tap_cb, group_lists, chain_pay, removed, chainW;
  dev_buf scan_scratch;
  prim::sort_scratch sort;
  // mr_records: where the latest result's rows and graph nodes are (its stamp, 0: none with a graph), and scratch;
  // mr_coords_records: where the latest result's rows are (rows_stamp, 0: none), for results with or without a graph
  uint64_t stamp = 0, graph_stamp = 0, rows_stamp = 0;
  graph_args last_graph;
  rows_args last_coords;
  uint64_t last_rows = 0;
  int last_max_rows = 0;
  dev_buf rec_cand, rec_i32, rec_f64, rec_info, rec_lines, rec_linf, rec_names, rec_text;
  pinned_buf rec_names_host;
  std::vector<pinned_buf*> text_pool;       // pinned slabs of mr_text, recycled like the result slabs
  std::vector<pinned_buf*> pinned_pool;     // result slabs are recycled: cudaMallocHost costs milliseconds
  std::mutex pool_mutex;                    // mr_result_free may run on another host thread than mr_align_batch
  std::vector<mr_staged*> staged_pool;      // device input buffers of staged batches, recycled (cudaMalloc synchronises the device)
  ~mr_workspace() { for(auto p : pinned_pool) delete p; for(auto p : text_pool) delete p; for(auto s : staged_pool) delete s; }
};

// text printed on the device (mr_records, mr_coords_records), in a pinned slab of the context's pool
struct mr_text {
  mr_context* ctx = nullptr;
  pinned_buf* host = nullptr;
  uint64_t size = 0;
};
// records.cu, shared by the two printers: the reads' names on the device (through a pinned staging buffer of the
// workspace; *d_off: nreads + 1 offsets from 0, *d_names: the bytes), and a slab of the pool for `bytes` of text
int upload_read_names(mr_context* ctx, mr_workspace& ws, const char* names, const uint64_t* name_off, uint32_t nreads,
                      const uint64_t** d_off, const char** d_names);
int take_text_slab(mr_context* ctx, mr_workspace& ws, mr_text* t, uint64_t bytes);

struct mr_result {
  mr_context* ctx = nullptr;
  uint64_t stamp = 0;               // mr_workspace::stamp of the batch that made it
  pinned_buf* host = nullptr;       // one pinned slab holding every array of the view (from the context's pool)
  mr_result_view view;
  // taps
  std::vector<int64_t>  tap_groups;
  std::vector<int32_t>  tap_offsets;
  std::vector<uint32_t> tap_lis;
};


// ---- chaining (chain.cu) ---------------------------------------------------------------------
struct chain_buffers {
  int32_t*  Lpb;  int32_t* Lsr;  uint32_t* Llen;  uint32_t* Lelt;   // indexed gs + array slot (global-memory tier)
  uint32_t* pprev; uint32_t* cstart;                                  // indexed gs + element
  int32_t*  Lwpb; int32_t* Lwsr;                                      // --window-size > 1: the window's base per list entry
};

struct survivors {
  // unsorted survivor rows (capacity cap); slot taken with atomicAdd on *count
  int32_t  *rs, *re, *qs, *qe, *nb_mers;
  uint32_t *pb_cons, *sr_cons, *pb_cover, *sr_cover, *ql, *sr, *read, *info_len;
  uint8_t  *rn, *use_bwd;
  double   *stretch, *offset, *avg_err;
  uint64_t *chain_pos;
  uint32_t *iter;           // --max-match round that produced the row (0 without it)
  uint64_t cap;
  unsigned long long* count;
  unsigned long long* info_total;
  uint32_t* read_cnt;
};

struct chain_args {
  index_view iv;
  const uint32_t* sr_len;            // length of every super-read, by global index (all parts)
  const uint64_t* keys; const uint64_t* pays; const uint64_t* group_start; uint64_t ngroups;
  const uint64_t* read_start;
  chain_buffers cb;
  double a, b, C, matching_mers, matching_bases;
  int forward;
  uint32_t unitigs_k, n_unitigs;
  const uint32_t* unitig_ids; const uint64_t* unitig_off;
  survivors sv;
  uint2* tap_lens; uint32_t* tap_cf; uint32_t* tap_cb; uint32_t* tap_sub;
  // filled by launch_chain: per-group verdict (chain length | fwd << 31) and the list of long chains
  uint32_t* group_nb; uint32_t* long_list; uint32_t* long_count; uint32_t* long_cursor;
  uint64_t* chain_pay;      // per group, at its slice: the chain's (pb, sr) pairs in chain order
  int max_match; uint8_t* removed;   // --max-match: hits already used by an emitted chain
  // fine pass (fine_aligner.cc:38-51): groups are the windows of the coarse rows, possibly empty
  uint32_t align_k;                  // mer length the coords are computed with (0: the index's k)
  int no_filter;                     // every group yields a row
  const uint32_t *group_read, *group_sr, *group_iter;   // identity of group g when not taken from keys[]
  uint32_t* dbg_cycles;              // MR_TRACE: SM cycles spent chaining each group
  uint32_t window;                   // --window-size (lis_align.hpp:17-45): 1 for every pipeline script
};
int launch_chain(mr_context* ctx, chain_args A, dev_buf& lists);

struct mr_workspace;
int launch_graph(mr_context* ctx, mr_workspace& ws, graph_args a, uint64_t S, int max_rows);
// rows per read above which the per-read kernels (coords order, overlap graph) use a CTA instead of a
// warp; MR_BIG_ROWS lowers it so that the tests drive the small fixtures through the CTA kernels
// rows of a read whose sequential graph state (33 bytes per row) still goes to shared memory: 6144 rows = 198 KB
// of the 227 KB a CTA may have on B200; larger reads use global scratch.  MR_HUGE_ROWS lowers it (tests).
inline int path_smem_rows_limit() {
  static const int v = [] { const char* e = getenv("MR_HUGE_ROWS"); const int x = e ? atoi(e) : 0; return x > 0 ? std::min(x, 6144) : 6144; }();
  return v;
}
// rows of a read up to which the per-read orderings (coords order, graph nodes) are a bitonic sort in shared
// memory instead of a ranking by counting; a power of two.  MR_SORT_ROWS lowers it (tests reach the fallback).
inline int big_sort_rows_limit() {
  static const int v = [] { const char* e = getenv("MR_SORT_ROWS"); int x = e ? atoi(e) : 0; if(x <= 0 || x > 4096) x = 4096;
                            int p = 1; while(p * 2 <= x) p *= 2; return p; }();
  return v;
}
inline int big_rows_threshold() {
  static const int v = [] { const char* e = getenv("MR_BIG_ROWS"); const int x = e ? atoi(e) : 0; return x > 0 ? x : 96; }();
  return v;
}

// C ABI over the host pipeline, for bench.py and tests: load inputs once, then run whole read sets
// through mr_align_batch (host buffers in, text out) exactly as the create_mega_reads tool does.
#include <atomic>
#include <chrono>
#include <cstring>
#include <iostream>
#include <stdexcept>

#include "pipeline.hpp"
#include "../records_common.hpp"

namespace {
struct tool {
  mrh::super_reads SR;
  mrh::unitigs     U;
  mrh::device_set  DS;
  mrh::device_unitigs DU;                             // the -u sequences on the device
  mrh::graph_options G;
  mr_params        P;
  std::vector<std::unique_ptr<mrh::read_batch>> batches;
  uint64_t total_bases = 0, total_reads = 0;
  std::string error;
  uint64_t last_text_bytes = 0, last_d2h_bytes = 0, last_h2d_bytes = 0, last_coords = 0;
  uint64_t last_lookups = 0, last_hits = 0, last_groups = 0;
  double   last_align_s = 0, last_format_s = 0;       // busy time of the two pipeline stages
};
}

extern "C" {

void* mrh_tool_create(const char* sr_fasta, const char* unitigs_path, int unitigs_is_fasta, unsigned mer, unsigned psa_min,
                      unsigned unitig_k, int device, char* err, size_t err_cap) {
  std::unique_ptr<tool> t(new tool);
  try {
    if(unitigs_is_fasta) t->U.load_sequences(unitigs_path); else t->U.load_lengths(unitigs_path);
    t->SR.append_fasta(sr_fasta);
    mrh::build_indexes(t->DS, std::vector<int>(1, device), t->SR, t->U, psa_min, mer);
    mrh::add_streams(t->DS, mrh::streams_per_device());
    mr_params_default(&t->P);
    t->P.unitigs_k = unitig_k;
    t->P.run_graph = 1;
    t->G.k_len = unitig_k;
    t->DU.upload(t->DS, t->U);
    return t.release();
  } catch(std::exception& e) {
    if(err && err_cap) { strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
    return nullptr;
  }
}

void mrh_tool_destroy(void* p) {
  tool* t = (tool*)p;
  if(!t) return;
  for(auto& b : t->batches) { mr_host_unpin(t->DS.ctx[0], b->codes.data()); mr_host_unpin(t->DS.ctx[0], b->nmask.data()); }
  delete t;
}

const char* mrh_tool_error(void* p) { return ((tool*)p)->error.c_str(); }
mr_context* mrh_tool_context(void* p) { return ((tool*)p)->DS.ctx[0]; }
// the tool keeps MR_STREAMS contexts on its device (batches in flight); all of them read the one index
unsigned mrh_tool_nstreams(void* p) { return (unsigned)((tool*)p)->DS.ctx.size(); }
mr_context* mrh_tool_stream_context(void* p, unsigned s) { return ((tool*)p)->DS.ctx[s]; }
mr_index* mrh_tool_index(void* p) { return ((tool*)p)->DS.idx[0]; }
mr_params* mrh_tool_params(void* p) { return &((tool*)p)->P; }
uint64_t mrh_tool_sr_bases(void* p) { return ((tool*)p)->SR.n; }
uint64_t mrh_tool_sr_count(void* p) { return ((tool*)p)->SR.nseq(); }

// loads (at most max_reads of) a read file into page-locked batches of ~batch_bases
int64_t mrh_tool_load_reads(void* p, const char* path, uint64_t batch_bases, uint64_t max_reads) {
  tool* t = (tool*)p;
  try {
    mrh::read_stream rs(std::vector<std::string>(1, path));
    while(max_reads == 0 || t->total_reads < max_reads) {
      std::unique_ptr<mrh::read_batch> b(new mrh::read_batch);
      b->clear();
      const uint64_t left = max_reads ? max_reads - t->total_reads : (1u << 20);
      if(!rs.next_batch(*b, batch_bases, (uint32_t)std::min<uint64_t>(left, 1u << 20), true)) break;   // parsed and packed
      t->total_bases += b->bases.size();
      t->total_reads += b->nreads();
      if(!b->packed()) b->pack();                   // the form the batch travels in (parsing + packing happen once, here)
      mr_host_pin(t->DS.ctx[0], b->codes.data(), b->codes.size() * 8);
      mr_host_pin(t->DS.ctx[0], b->nmask.data(), b->nmask.size() * 8);
      t->batches.push_back(std::move(b));
    }
    return (int64_t)t->total_bases;
  } catch(std::exception& e) { t->error = e.what(); return -1; }
}
uint64_t mrh_tool_nbatches(void* p) { return ((tool*)p)->batches.size(); }
uint64_t mrh_tool_nreads(void* p) { return ((tool*)p)->total_reads; }
// batch accessors, so a caller can stage the same batches on the device itself
const char* mrh_tool_batch_bases(void* p, uint64_t i, uint64_t* nbytes) {
  tool* t = (tool*)p; *nbytes = t->batches[i]->bases.size(); return t->batches[i]->bases.data();
}
const uint64_t* mrh_tool_batch_codes(void* p, uint64_t i, uint64_t* nwords) {
  tool* t = (tool*)p; *nwords = t->batches[i]->codes.size(); return t->batches[i]->codes.data();
}
const uint64_t* mrh_tool_batch_nmask(void* p, uint64_t i, uint64_t* nwords) {
  tool* t = (tool*)p; *nwords = t->batches[i]->nmask.size(); return t->batches[i]->nmask.data();
}
const uint64_t* mrh_tool_batch_starts(void* p, uint64_t i, uint32_t* nreads) {
  tool* t = (tool*)p; *nreads = t->batches[i]->nreads(); return t->batches[i]->start.data();
}

// One full pass over the loaded reads through the public path: mr_align_batch from host memory
// (H2D inside), results back (D2H inside), text records printed on the device (mr_records) right after each
// batch and written by a second thread while the next batch is already on the GPU (the same stages as the
// command line tools).  `threads` is accepted for compatibility; nothing is formatted on the host.
// out_path may be null/empty (text is produced and dropped).  Returns read bases processed, <0 on error.
// mrh_tool_run_range: the same over batches [first, first + count) only (bench.py's parity gate writes
// the records of the reads the CPU reference was run on).
int64_t mrh_tool_run_range(void* p, unsigned threads, const char* out_path, uint64_t first, uint64_t count) {
  tool* t = (tool*)p;
  if(first > t->batches.size()) first = t->batches.size();
  count = std::min<uint64_t>(count, t->batches.size() - first);
  FILE* out = nullptr;
  if(out_path && *out_path) { out = fopen(out_path, "w"); if(!out) { t->error = "cannot open output"; return -1; } }
  t->last_text_bytes = t->last_d2h_bytes = t->last_h2d_bytes = t->last_coords = 0;
  t->last_lookups = t->last_hits = t->last_groups = 0;
  t->last_align_s = t->last_format_s = 0;
  // one aligner thread per context takes the next batch; results are formatted in batch order
  const size_t nb = (size_t)count;
  std::vector<mr_result*> done(nb, nullptr);
  std::vector<mr_text*> texts(nb, nullptr);
  uint64_t bases_done = 0;
  std::vector<char> ready(nb, 0);
  std::mutex m;
  std::condition_variable cv;
  size_t formatted = 0;                       // batches the formatter is done with (guarded by m)
  bool   stop = false;
  std::string error, align_error;
  std::thread formatter([&]() {
    mrh::background_thread();
    for(size_t i = 0; i < nb; ++i) {
      mr_result* r = nullptr;
      mr_text* text = nullptr;
      {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { return ready[i] || stop; });
        if(!ready[i]) return;
        r = done[i]; text = texts[i];
      }
      const auto f0 = std::chrono::steady_clock::now();
      mrh::read_batch* b = t->batches[first + i].get();
      bases_done += b->bases.size();
      mr_result_view v;
      mr_result_get(r, &v);
      const char* bytes = nullptr;
      uint64_t nbytes = 0;
      mr_text_get(text, &bytes, &nbytes);
      if(out && nbytes && fwrite(bytes, 1, nbytes, out) != nbytes) error = "write error on output file";
      t->last_text_bytes += nbytes;
      t->last_d2h_bytes += nbytes;
      mr_text_free(text);
      t->last_h2d_bytes += (b->codes.size() + b->nmask.size() + b->nreads() + 1) * 8ULL;
      uint64_t info = 0;
      for(uint64_t c = 0; c < v.ncoords; ++c) info += v.info_len[c];
      t->last_d2h_bytes += (v.nreads + 1) * 8ULL + v.ncoords * (5 * 4 + 6 * 4 + 2 + 3 * 8 + 8 + 4 + 2 + 5 * 4) + info * 8;
      t->last_coords += v.ncoords;
      t->last_lookups += v.n_kmers_looked_up; t->last_hits += v.n_hits; t->last_groups += v.n_groups;
      mr_result_free(r);
      t->last_format_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - f0).count();
      { std::lock_guard<std::mutex> l(m); formatted = i + 1; }
      cv.notify_all();
    }
  });
  std::atomic<size_t> next(0);
  std::vector<double> busy(t->DS.ctx.size(), 0.0);
  std::vector<std::thread> aligners;
  for(size_t s = 0; s < t->DS.ctx.size(); ++s) {
    aligners.emplace_back([&, s]() {
      while(true) {
        const size_t i = next++;
        if(i >= nb) break;
        {   // stay at most a few batches ahead of the formatter (bounds the pinned result memory)
          std::unique_lock<std::mutex> l(m);
          cv.wait(l, [&] { return i < formatted + 3 + t->DS.ctx.size() || stop; });
          if(stop) break;
        }
        mr_result* r = nullptr;
        const auto a0 = std::chrono::steady_clock::now();
        mrh::read_batch* b = t->batches[first + i].get();
        const int rc = mr_align_batch_packed(t->DS.ctx[s], t->DS.idx[s], &t->P, b->codes.data(), b->nmask.data(), b->start.data(), b->nreads(), &r);
        mr_text* text = nullptr;
        std::string rec_error;
        if(rc == MR_OK) {
          try { text = mrh::device_records(t->DS.ctx[s], r, mrh::records_params(t->G), t->DU.of(t->DS.ctx[s]), b->name); }
          catch(std::exception& e) { rec_error = e.what(); mr_result_free(r); }
        }
        busy[s] += std::chrono::duration<double>(std::chrono::steady_clock::now() - a0).count();
        std::lock_guard<std::mutex> l(m);
        if(rc != MR_OK || !rec_error.empty()) {
          if(align_error.empty()) align_error = rc != MR_OK ? mr_last_error(t->DS.ctx[s]) : rec_error;
          stop = true; cv.notify_all(); break;
        }
        done[i] = r; texts[i] = text; ready[i] = 1;
        cv.notify_all();
      }
    });
  }
  for(auto& th : aligners) th.join();
  formatter.join();
  for(double b : busy) t->last_align_s = std::max(t->last_align_s, b);
  for(size_t i = 0; i < nb; ++i) if(ready[i] && i >= formatted) { mr_text_free(texts[i]); mr_result_free(done[i]); }   // only after an error
  if(out) fclose(out);
  if(!align_error.empty() || !error.empty()) { t->error = align_error.empty() ? error : align_error; return -1; }
  return (int64_t)bases_done;
}
int64_t mrh_tool_run(void* p, unsigned threads, const char* out_path) {
  return mrh_tool_run_range(p, threads, out_path, 0, ~0ULL);
}
// Parses read files the way the tools do and returns what came out, for tests that have no GPU: out6 = { reads, bases,
// FNV-1a of the bases, FNV-1a of the names (each followed by a newline), FNV-1a of the packed code words covering the
// bases, number of non-ACGT characters according to the mask }.  Returns 0, or -1 with the message in err.
int mrh_selftest_read_stream(const char* const* paths, unsigned npaths, uint64_t batch_bases, unsigned threads, uint64_t* out6,
                             char* err, size_t err_cap) {
  try {
    std::vector<std::string> ps(paths, paths + npaths);
    mrh::read_stream rs(ps, threads);
    uint64_t h_bases = 1469598103934665603ULL, h_names = h_bases, h_codes = h_bases, reads = 0, bases = 0, nonacgt = 0;
    auto fnv = [](uint64_t h, const void* p, size_t n) { const unsigned char* b = (const unsigned char*)p; for(size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ULL; } return h; };
    while(true) {
      mrh::read_batch b;
      b.clear();
      if(!rs.next_batch(b, batch_bases, 1u << 20, true)) break;
      reads += b.nreads(); bases += b.bases.size();
      h_bases = fnv(h_bases, b.bases.data(), b.bases.size());
      for(const auto& n : b.name) { h_names = fnv(h_names, n.data(), n.size()); h_names = fnv(h_names, "\n", 1); }
      for(uint64_t g = 0; g < b.bases.size(); ++g) {          // the packed form, base by base (independent of batch cuts)
        const unsigned char code = (unsigned char)((b.codes[g >> 5] >> (2 * (g & 31))) & 3);
        const unsigned char bad = (unsigned char)((b.nmask[g >> 6] >> (g & 63)) & 1);
        const unsigned char both = (unsigned char)(code | (bad << 2));
        h_codes = fnv(h_codes, &both, 1);
        nonacgt += bad;
      }
      if(b.start.size() != (size_t)b.nreads() + 1 || b.start.back() != b.bases.size()) throw std::runtime_error("inconsistent batch");
    }
    out6[0] = reads; out6[1] = bases; out6[2] = h_bases; out6[3] = h_names; out6[4] = h_codes; out6[5] = nonacgt;
    return 0;
  } catch(std::exception& e) {
    if(err && err_cap) { strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
    return -1;
  }
}
uint64_t mrh_selftest_fixed_format(uint64_t samples, uint64_t seed) { return mrh::selftest_fixed_format(samples, seed); }
// The fixed-point formatter of the records (records_common.hpp) and printf, side by side: both strings of x with d
// decimals; returns whether they are equal.
int mrh_fixed_format_pair(double x, int d, char* mine, char* libc) {
  const int n = mrfmt::fmt_fixed(mine, x, d);
  mine[n] = 0;
  snprintf(libc, mrfmt::kFixedMax + 8, "%.*f", d, x);
  return strcmp(mine, libc) == 0;
}
// The device's std::sort port against std::sort on n elements whose keys (kind 0, 1: ints, compared as the greedy
// and maximal tilings compare lpath and tiling_end; 2: doubles, as the weighted tiling compares weights) are keys[];
// returns the number of positions where the two permutations differ.
uint64_t mrh_selftest_sort(int kind, const double* keys, uint64_t n) {
  std::vector<int> a(n), b(n);
  for(uint64_t i = 0; i < n; ++i) a[i] = b[i] = (int)i;
  auto run = [&](auto comp) { std::sort(a.begin(), a.end(), comp); mrfmt::std_sort(b.data(), (long)n, comp); };
  if(kind == 0) run([&](int i, int j) { return (int)keys[j] < (int)keys[i]; });
  else if(kind == 1) run([&](int i, int j) { return keys[i] < keys[j]; });
  else run([&](int i, int j) { return keys[j] < keys[i]; });
  uint64_t bad = 0;
  for(uint64_t i = 0; i < n; ++i) bad += a[i] != b[i];
  return bad;
}
// The host formatter (mrh::format_mega_reads, the reference of the device printer) over a result: the super-read
// paths the result's rows index (CSR), the k-unitig lengths, the sequences (useq == NULL: -l), the reads' names and
// lengths (read_start: nreads + 1 offsets) and the printing options.  *out: malloc'ed text (mrh_free).  Returns 0,
// or -1 with the message the tools print in err.
int mrh_format_records(const mr_result* r, const uint32_t* path_ids, const uint64_t* path_off, uint32_t npaths,
                       const int32_t* ulen, uint32_t nu, const char* useq, const uint64_t* uoff,
                       const char* names, const uint64_t* name_off, const uint64_t* read_start,
                       const mr_records_params* p, char** out, uint64_t* size, char* err, size_t err_cap) {
  try {
    mr_result_view v;
    if(mr_result_get(r, &v) != MR_OK || !v.lstart) throw std::runtime_error("the result has no overlap graph");
    mrh::super_reads sr;
    sr.unitig_off.assign(path_off, path_off + npaths + 1);
    sr.unitig_ids.assign(path_ids, path_ids + path_off[npaths]);
    mrh::unitigs u;
    u.len.assign(ulen, ulen + nu);
    if(useq) {
      u.off.assign(uoff, uoff + nu + 1);
      u.fwd.assign(useq, uoff[nu]);
      u.rc.resize(u.fwd.size());
      for(uint32_t i = 0; i < nu; ++i)
        for(uint64_t j = 0, n = uoff[i + 1] - uoff[i]; j < n; ++j) u.rc[uoff[i] + j] = mrfmt::revcomp_base((unsigned char)useq[uoff[i] + n - 1 - j]);
    }
    mrh::read_batch b;
    b.start.assign(read_start, read_start + v.nreads + 1);
    for(uint32_t i = 0; i < v.nreads; ++i) b.name.emplace_back(names + name_off[i], name_off[i + 1] - name_off[i]);
    mrh::graph_options o;
    o.k_len = p->unitigs_k; o.overlap_play = p->overlap_play; o.density = p->density; o.min_length = p->min_length;
    o.tiling = p->tiling; o.trim = p->trim;
    mrh::text_buf text;
    mrh::format_mega_reads(v, b, 0, v.nreads, sr, u, o, text);
    *out = (char*)malloc(text.size() + 1);
    if(!*out) throw std::bad_alloc();
    if(text.size()) memcpy(*out, text.data(), text.size());
    *size = text.size();
    return 0;
  } catch(std::exception& e) {
    if(err && err_cap) { strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
    return -1;
  }
}
// The host coords formatter (mrh::format_coords, the reference of the device printer and the tool's --details path)
// over a result: the super-reads' names and unitig paths (CSR, path_ids may be NULL when all paths are empty), the
// reads' names and lengths (read_start: nreads + 1 offsets), --compact and -0.  *out: malloc'ed text (mrh_free).
// Returns 0, or -1 with the message in err.
int mrh_format_coords(const mr_result* r, const char* sr_names, const uint64_t* sr_name_off, const uint32_t* path_ids,
                      const uint64_t* path_off, uint32_t nseq, const char* names, const uint64_t* name_off,
                      const uint64_t* read_start, int compact, int zero_match, char** out, uint64_t* size, char* err, size_t err_cap) {
  try {
    mr_result_view v;
    if(mr_result_get(r, &v) != MR_OK) throw std::runtime_error("no result");
    mrh::super_reads sr;
    for(uint32_t i = 0; i < nseq; ++i) sr.name.emplace_back(sr_names + sr_name_off[i], sr_name_off[i + 1] - sr_name_off[i]);
    sr.unitig_off.assign(path_off, path_off + nseq + 1);
    if(path_ids) sr.unitig_ids.assign(path_ids, path_ids + path_off[nseq]);
    for(uint64_t i = 0; i < v.ncoords; ++i)
      if(v.sr[i] >= nseq) throw std::runtime_error("a row refers to a super-read that the names do not have");
    mrh::read_batch b;
    b.start.assign(read_start, read_start + v.nreads + 1);
    for(uint32_t i = 0; i < v.nreads; ++i) b.name.emplace_back(names + name_off[i], name_off[i + 1] - name_off[i]);
    mrh::text_buf text;
    mrh::format_coords(v, b, 0, v.nreads, sr, compact != 0, zero_match == 0, text);
    *out = (char*)malloc(text.size() + 1);
    if(!*out) throw std::bad_alloc();
    if(text.size()) memcpy(*out, text.data(), text.size());
    *size = text.size();
    return 0;
  } catch(std::exception& e) {
    if(err && err_cap) { strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
    return -1;
  }
}
// The "%g" formatter of the coords lines (records_common.hpp) and printf, side by side: both strings of x; returns
// whether they are equal.  Each buffer holds at least mrfmt::kGeneralMax + 1 bytes.
int mrh_general_format_pair(double x, char* mine, char* libc) {
  const int n = mrfmt::fmt_general(mine, x);
  mine[n] = 0;
  snprintf(libc, mrfmt::kGeneralMax + 1, "%g", x);
  return strcmp(mine, libc) == 0;
}
void mrh_free(void* p) { free(p); }
void mrh_tool_stage_seconds(void* p, double* align_s, double* format_s) {
  tool* t = (tool*)p; *align_s = t->last_align_s; *format_s = t->last_format_s;
}
void mrh_tool_last_stats(void* p, uint64_t* out8) {
  tool* t = (tool*)p;
  out8[0] = t->last_text_bytes; out8[1] = t->last_h2d_bytes; out8[2] = t->last_d2h_bytes; out8[3] = t->last_coords;
  out8[4] = t->last_lookups; out8[5] = t->last_hits; out8[6] = t->last_groups; out8[7] = t->total_bases;
}

} // extern "C"

// Host side of the B200 mega-reads tools: input parsing (super-read FASTA, k-unitig files,
// long-read FASTA/FASTQ streams), 2-bit packing, and the per-read post-processing that turns the
// device's coords / graph rows into the reference's text records.  Plain C++17, no CUDA; the
// device is reached only through include/mega_reads_b200.h.
#pragma once
#include <functional>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "mega_reads_b200.h"

namespace mrh {

// ---- super-reads: sequence_psa::append_fasta (superread_parser.cc:12-46) + frag_info (frag_info.hpp:18-35)
struct super_reads {
  std::vector<uint64_t>    text2bit;     // compact_dna layout
  uint64_t                 n = 0;
  std::vector<uint64_t>    start;        // nseq + 1
  std::vector<std::string> name;         // header line after '>'
  std::vector<uint32_t>    unitig_ids;   // CSR of forward paths, (id << 1) | (ori == 'R')
  std::vector<uint64_t>    unitig_off;   // nseq + 1
  uint32_t nseq() const { return (uint32_t)name.size(); }
  void append_fasta(const std::string& path);          // throws std::runtime_error like the reference
  // unitig path of super-read s in the orientation a coords row uses it
  uint32_t path_len(uint32_t s) const { return (uint32_t)(unitig_off[s + 1] - unitig_off[s]); }
  uint32_t path_at(uint32_t s, bool bwd, uint32_t t) const {
    const uint64_t b = unitig_off[s], e = unitig_off[s + 1];
    return bwd ? (unitig_ids[e - 1 - t] ^ 1u) : unitig_ids[b + t];
  }
  std::string row_name(uint32_t s, bool bwd) const;   // fwd.name / bwd.name of frag_info
};

// ---- k-unitigs: read_unitigs_lengths / read_unitigs_sequences (misc.cc:11-37)
struct unitigs {
  std::vector<int32_t>     len;
  // only with -u: every sequence back to back in one arena, and the reverse complements
  // (rev_comp_ of super_read_name.cc:106-114, built once at load) in a second one with the same offsets.
  // Printing a mega-read copies ~20 unitigs of ~500 bases: with one heap string per unitig every piece cost
  // two dependent cache misses before the copy could start; an offset table that fits the L2 and
  // contiguous text (prefetched one piece ahead) make the copy run at memcpy speed.
  std::string              fwd, rc;
  std::vector<uint64_t>    off;          // len.size() + 1 offsets into fwd / rc
  bool has_sequences() const { return !off.empty(); }
  const char* sequence(uint32_t id, bool reversed) const { return (reversed ? rc.data() : fwd.data()) + off[id]; }
  void load_lengths(const std::string& path);
  void load_sequences(const std::string& path);
};

// ---- long reads: jellyfish::whole_sequence_parser as used in create_mega_reads.cc:51-58
struct read_batch {
  std::string              bases;        // concatenated
  std::vector<uint64_t>    start;        // nreads + 1
  std::vector<std::string> name;         // header up to the first white space
  // what travels to the GPU: 2 bits per base + a mask of the non-ACGT characters (mr_pack_reads), 0.375 bytes per base
  std::vector<uint64_t>    codes, nmask;
  uint32_t nreads() const { return (uint32_t)name.size(); }
  void clear() { bases.clear(); start.assign(1, 0); name.clear(); codes.clear(); nmask.clear(); }
  // The pipeline page-locks the packed arrays of the batches it recycles (plain DMA instead of a staged copy);
  // before_regrow is its hook to unlock them before a resize moves them.
  std::function<void(read_batch&)> before_regrow;
  const void* locked[2] = { nullptr, nullptr };
  void size_packed(uint64_t cwords, uint64_t mwords) {
    if((cwords > codes.capacity() || mwords > nmask.capacity()) && before_regrow) before_regrow(*this);
    codes.resize(cwords); nmask.resize(mwords);
  }
  void pack() {
    size_packed(mr_packed_code_words(bases.size()), mr_packed_mask_words(bases.size()));
    mr_pack_reads(bases.data(), bases.size(), codes.data(), nmask.data());
  }
  bool packed() const { return !nmask.empty(); }
};
// Reads FASTA / FASTQ files batch by batch.  A regular file is mapped and scanned in place, anything else (a FIFO,
// a process substitution: mega_reads_assemble_cluster2.sh:472) is read in large chunks -- the stream is never
// seeked.  A batch is cut in two steps: a serial scan that only finds the lines (memchr) and notes where each
// record's sequence pieces lie, then `threads` workers that copy the pieces into the batch and pack it
// (mr_pack_reads_range) -- parsing 0.6 GB of reads per step must not take longer than aligning them.
class read_stream {
  struct piece { uint64_t src; uint32_t len; uint64_t dst; };      // src: offset into the window
  std::vector<std::string> paths_;
  size_t next_path_ = 0;
  // the window: either the mapped file or the bytes read so far that are not consumed yet
  const char* win_ = nullptr;
  size_t win_len_ = 0, pos_ = 0;
  void*  map_ = nullptr;
  size_t map_len_ = 0;
  int    fd_ = -1;
  std::vector<char> buf_;
  bool   eof_ = true, open_ = false;
  char   kind_ = 0;                       // '>' or '@': format of the current file
  unsigned threads_;
  std::vector<piece> pieces_;
  // records of a mapped FASTA file found ahead of the batches, by all threads at once (prescan)
  struct prerec { uint64_t name_b; uint32_t name_len; uint32_t npieces; uint64_t first_piece, len, end_pos; };
  std::vector<prerec> pre_;
  std::vector<piece>  pre_pieces_;
  size_t pre_next_ = 0;
  bool prescan();
  bool open_next();
  void close_current();
  bool refill();                          // stream mode: more bytes behind the window; false at end of file
  // scans one record starting at pos_; 1: done, 0: the window ends inside it (refill and try again), -1: end of file
  int scan_record(read_batch& b, uint64_t& nbases);
public:
  explicit read_stream(const std::vector<std::string>& paths, unsigned threads = 0);
  ~read_stream() { close_current(); }
  read_stream(const read_stream&) = delete;
  read_stream& operator=(const read_stream&) = delete;
  // appends reads until the batch holds >= max_bases bases or max_reads reads; false when exhausted.
  // with pack, the batch also comes out packed (read_batch::codes / nmask)
  bool next_batch(read_batch& b, uint64_t max_bases, uint32_t max_reads, bool pack = false);
};

// ---- output text.  A batch of mega-read records is tens of megabytes that are written once and read
// once (by fwrite): a growable byte buffer that never zero-fills or re-copies its storage.  (Streaming
// stores for the unitig sequences were measured too: faster in isolation, slower here, where the
// buffers of a batch are reused and stay in the last-level cache.)
// lowers the calling thread's priority below the threads that feed the GPUs (host_common.cpp)
void background_thread();

class text_buf {
  char*  p_ = nullptr;
  size_t size_ = 0, cap_ = 0;
  void grow(size_t need);
public:
  text_buf() = default;
  text_buf(const text_buf&) = delete;
  text_buf& operator=(const text_buf&) = delete;
  text_buf(text_buf&& o) noexcept : p_(o.p_), size_(o.size_), cap_(o.cap_) { o.p_ = nullptr; o.size_ = o.cap_ = 0; }
  text_buf& operator=(text_buf&& o) noexcept { if(this != &o) { release(); p_ = o.p_; size_ = o.size_; cap_ = o.cap_; o.p_ = nullptr; o.size_ = o.cap_ = 0; } return *this; }
  ~text_buf() { release(); }
  void release();
  const char* data() const { return p_; }
  size_t size() const { return size_; }
  size_t capacity() const { return cap_; }
  bool empty() const { return size_ == 0; }
  void clear() { size_ = 0; }
  void reserve(size_t n) { if(n > cap_) grow(n); }
  void append(const char* s, size_t n);
  char* grab(size_t n) { if(size_ + n > cap_) grow(size_ + n); char* w = p_ + size_; size_ += n; return w; }   // n bytes for the caller to fill
  void flush();
  text_buf& operator+=(char c) { if(size_ + 1 > cap_) grow(size_ + 1); p_[size_++] = c; return *this; }
  text_buf& operator+=(const char* s) { append(s, strlen(s)); return *this; }
  text_buf& operator+=(const std::string& s) { append(s.data(), s.size()); return *this; }
};

// ---- options shared by the two tools (Appendix B of SURVEY.md; create_mega_reads_cmdline.yaggo)
struct graph_options {
  double   overlap_play = 1.3;
  uint32_t k_len = 0;
  double   density = 0.029, min_length = 100.0;
  int      tiling = 1;      // 0 none, 1 greedy, 2 maximal, 3 weighted
  int      trim = 0;        // 0 none, 1 match, 2 branch (== match)
};

// Text records of create_mega_reads for reads [r0, r1) of a result (overlap_graph.cc:61-299,
// overlap_graph.hpp:198-262): best terminal node per component, tiling, one line per mega-read.  The tools print
// their records on the device (mr_records); this host formatter is the one for --dot, whose edges it recomputes,
// and the reference the device printer is tested against.
// dot: when not null, also the reference's --dot text for these reads (overlap_graph.hpp:189-196, overlap_graph.cc:49-50,
// 133-146,271): one "digraph" per read with every node, every overlap edge (recomputed here from the rows: the device
// keeps only what the longest paths need) and the edges of the printed paths in red.  dot_state carries the one
// piece of stream state the reference's output depends on (the first node of the stream prints its implied
// positions with 6 decimals, every later one with 2).
struct dot_state { bool first_node = true; double errors = 3.0; int bases = 0; };
void format_mega_reads(const mr_result_view& v, const read_batch& batch, uint32_t r0, uint32_t r1,
                       const super_reads& sr, const unitigs& u, const graph_options& o, text_buf& out,
                       text_buf* dot = nullptr, dot_state* ds = nullptr);
// self test of the fixed-point number formatter behind the mega-read lines (records_common.hpp): `samples`
// pseudo-random doubles (decimal grids, half-way points, binary fractions, wide exponent range), "%.2f" and
// "%.4f", against the C library; returns the number of strings that differ (must be 0)
uint64_t selftest_fixed_format(uint64_t samples, uint64_t seed);

// jf_aligner coords records (jf_aligner.cc:41-70).  The tool prints them on the device (mr_coords_records); this host
// formatter is the one for --details, and the reference the device printer is tested against.
void format_coords(const mr_result_view& v, const read_batch& batch, uint32_t r0, uint32_t r1, const super_reads& sr,
                   bool compact, bool zero_skip, text_buf& out);

// jf_aligner --details records (jf_aligner.cc:72-108): one line per (read, super-read) pair with every
// k-mer hit "pb:sr" in read order, the hits of the reported chain in brackets.  Needs the parity
// taps of the result (mr_context_keep_taps).
void format_details(const mr_result* r, const read_batch& batch, const super_reads& sr, text_buf& out);

// ---- compact coords files (jf_aligner --coords, format of print_coords, jf_aligner.cc:41-70),
// read back the way longest_path_overlap_graph2 does (coords_parsing.cc:7-64): records
// ">N read-name" + N rows; a row = 14 numbers, the super-read name (a unitig path), then one
// "mers:bases" pair per kmers_info entry.  One batch holds the rows of whole reads as the columns
// of an mr_result_view over its own vectors, ready for mr_graph_batch.
struct coords_batch {
  read_batch  reads;                    // names; start[] is the running sum of Rlen (no bases)
  std::vector<uint32_t> read_len;
  super_reads paths;                    // entry i: name and unitig path of row i
  std::vector<uint64_t> read_coords, info_off;
  std::vector<int32_t>  rs, re, qs, qe, nb_mers, kmers_info, bases_info;
  std::vector<uint32_t> pb_cons, sr_cons, pb_cover, sr_cover, ql, sr, info_len;
  std::vector<uint8_t>  rn, use_bwd;
  std::vector<double>   stretch, offset, avg_err;
  mr_result_view view() const;
  void clear();
};
class coords_file {
  FILE* f_ = nullptr;
  std::string line_;
  bool started_ = false, pending_ = false;
  bool getline();
public:
  explicit coords_file(const std::string& path);
  ~coords_file() { if(f_) fclose(f_); }
  // appends whole reads until the batch holds >= max_rows rows; false when the file is exhausted
  bool next_batch(coords_batch& b, uint64_t max_rows);
};

} // namespace mrh

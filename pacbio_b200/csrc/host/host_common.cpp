#include <cerrno>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <new>
#include <cstring>
#include "host_common.hpp"
#include "../records_common.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <exception>
#include <fstream>
#include <functional>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <map>
#include <stdexcept>
#include <thread>

namespace mrh {

// The threads that pack reads and print records yield to the ones that drive the GPUs: with few cores per GPU (32 for
// 8) the printing threads keep every core busy, and a thread that wakes up from a stream wait to launch the next
// kernels of a batch must not queue behind them -- every such wait is device idle time (8 GPUs: mr_align_batch took
// 2.7 times as long per batch as with one).  Raising one's own nice value needs no privilege.  MR_NICE=0 leaves the
// priorities alone, another value sets the increment.
void background_thread() {
  static const int inc = [] { const char* e = getenv("MR_NICE"); return e ? atoi(e) : 10; }();
  if(inc > 0) setpriority(PRIO_PROCESS, (id_t)syscall(SYS_gettid), inc);
}

// ================================================================================================
// output text
// ================================================================================================
void text_buf::release() { free(p_); p_ = nullptr; size_ = cap_ = 0; }
void text_buf::grow(size_t need) {
  size_t cap = std::max<size_t>(need + need / 4, 1 << 16);
  cap = (cap + 4095) & ~(size_t)4095;
  char* q = (char*)aligned_alloc(4096, cap);
  if(!q) throw std::bad_alloc();
  if(size_) memcpy(q, p_, size_);
  free(p_);
  p_ = q; cap_ = cap;
}
void text_buf::flush() { }
void text_buf::append(const char* s, size_t n) {
  if(size_ + n > cap_) grow(size_ + n);
  memcpy(p_ + size_, s, n);
  size_ += n;
}

// ================================================================================================
// super-reads
// ================================================================================================
// "12F_7R_3F" -> (id << 1) | ori.  Mirrors super_read_name::parse (super_read_name.cc:74-90): every
// '_'-separated piece must start with a number, the orientation is its last character ('R' or not);
// a piece without digits invalidates the whole name (empty path).
static bool parse_path(const std::string& name, std::vector<uint32_t>& out) {
  out.clear();
  if(name.empty()) return true;
  size_t pos = 0;
  while(true) {
    const size_t us = name.find('_', pos);
    const size_t end = us == std::string::npos ? name.size() : us;
    size_t d = pos;
    while(d < end && (name[d] == ' ' || name[d] == '\t')) ++d;     // std::stoul skips leading blanks
    if(d < end && name[d] == '+') ++d;
    uint64_t id = 0;
    size_t nd = 0;
    while(d < name.size() && name[d] >= '0' && name[d] <= '9') { id = id * 10 + (uint64_t)(name[d] - '0'); ++d; ++nd; }
    if(nd == 0) { out.clear(); return false; }
    const char ori = end > 0 ? name[end - 1] : 'F';
    out.push_back((uint32_t)((id & 0x7fffffffu) << 1) | (ori == 'R' ? 1u : 0u));
    if(us == std::string::npos) break;
    pos = us + 1;
  }
  return true;
}

void super_reads::append_fasta(const std::string& path) {
  std::ifstream is(path, std::ios::binary);
  if(!is.good()) throw std::runtime_error("Can't open file " + path);
  if(is.peek() != '>') throw std::runtime_error("Not in fasta format");
  if(start.empty()) { start.push_back(0); unitig_off.push_back(0); }
  std::string header, line;
  std::vector<uint32_t> upath;
  int c = is.peek();
  while(c != EOF) {
    std::getline(is, header);
    const uint64_t old = n;
    for(c = is.peek(); c != '>' && c != EOF; c = is.peek()) {
      std::getline(is, line);
      const uint64_t need = (n + line.size() + 31) / 32 + 1;
      if(text2bit.size() < need) text2bit.resize(std::max<uint64_t>(need, text2bit.size() * 2), 0);
      for(unsigned char x : line) {                                  // compact_dna.hpp:102-107 (SWAR mapping)
        const uint64_t code = ((x >> 1) ^ (x >> 2)) & 3;
        text2bit[n >> 5] |= code << (2 * (n & 31));
        ++n;
      }
    }
    if(n > old) {
      name.push_back(header.substr(1));
      parse_path(name.back(), upath);
      unitig_ids.insert(unitig_ids.end(), upath.begin(), upath.end());
      unitig_off.push_back(unitig_ids.size());
      start.push_back(n);
    }
  }
}

std::string super_reads::row_name(uint32_t s, bool bwd) const {
  const uint32_t u = path_len(s);
  if(!bwd || u == 0) return name[s];
  std::string r;
  for(uint32_t t = 0; t < u; ++t) {
    const uint32_t x = path_at(s, true, t);
    if(t) r += '_';
    r += std::to_string(x >> 1);
    r += (x & 1) ? 'R' : 'F';
  }
  return r;
}

// ================================================================================================
// k-unitigs
// ================================================================================================

void unitigs::load_lengths(const std::string& path) {
  std::ifstream is(path);
  if(!is.good()) throw std::runtime_error("Failed to open unitig lengths map file '" + path + "'");
  std::string id;
  unsigned int l;
  while(is >> id >> l) len.push_back((int32_t)l);
}

void unitigs::load_sequences(const std::string& path) {
  std::ifstream is(path, std::ios::binary);
  if(!is.good()) throw std::runtime_error("Failed to open unitigs sequence file '" + path + "'");
  std::string hdr, s;
  off.assign(1, 0);
  while(std::getline(is, hdr)) {
    if(!std::getline(is, s)) s.clear();
    len.push_back((int32_t)s.size());
    fwd += s;
    off.push_back(fwd.size());
  }
  // Printing a mega-read copies the unitigs of its path, reverse-complemented for 'R' entries;
  // doing the complement once here turns every later append into a memcpy.
  rc.resize(fwd.size());
  const unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  std::vector<std::thread> th;
  for(unsigned t = 0; t < nt; ++t)
    th.emplace_back([&, t]() {
      for(size_t i = t; i + 1 < off.size(); i += nt) {
        const char* f = fwd.data() + off[i];
        char* r = &rc[off[i]];
        const size_t n = off[i + 1] - off[i];
        for(size_t j = 0; j < n; ++j) r[j] = mrfmt::revcomp_base((unsigned char)f[n - 1 - j]);
      }
    });
  for(auto& x : th) x.join();
}

// ================================================================================================
// long reads
// ================================================================================================
read_stream::read_stream(const std::vector<std::string>& paths, unsigned threads)
  : paths_(paths), threads_(threads ? threads : std::max(1u, std::min(16u, std::thread::hardware_concurrency()))) { }

void read_stream::close_current() {
  if(map_) { munmap(map_, map_len_); map_ = nullptr; }
  if(fd_ >= 0) { close(fd_); fd_ = -1; }
  win_ = nullptr; win_len_ = 0; pos_ = 0; eof_ = true; open_ = false;
  buf_.clear();
  pre_.clear(); pre_pieces_.clear(); pre_next_ = 0;
}

bool read_stream::open_next() {
  close_current();
  if(next_path_ >= paths_.size()) return false;
  const std::string& p = paths_[next_path_++];
  fd_ = open(p.c_str(), O_RDONLY);
  if(fd_ < 0) throw std::runtime_error("Can't open file '" + p + "'");
  open_ = true; kind_ = 0;
  struct stat st;
  if(fstat(fd_, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
    void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd_, 0);
    if(m != MAP_FAILED) {
      map_ = m; map_len_ = (size_t)st.st_size;
      madvise(m, map_len_, MADV_SEQUENTIAL);
      win_ = (const char*)m; win_len_ = map_len_; pos_ = 0; eof_ = true;      // everything is in the window
      return true;
    }
  }
  eof_ = false;                              // stream mode: the window grows through refill()
  win_ = nullptr; win_len_ = 0; pos_ = 0;
  return true;
}

bool read_stream::refill() {
  if(eof_ || map_) return false;
  // drop what has been consumed only when no piece of the current batch points into it (the caller resets
  // pieces_ and pos_-relative offsets stay valid because offsets are into buf_, which is only appended to here)
  const size_t chunk = 64u << 20;
  const size_t old = buf_.size();
  buf_.resize(old + chunk);
  size_t got = 0;
  while(got < chunk) {
    const ssize_t r = read(fd_, buf_.data() + old + got, chunk - got);
    if(r < 0) { if(errno == EINTR) continue; throw std::runtime_error("read error on '" + paths_[next_path_ - 1] + "'"); }
    if(r == 0) { eof_ = true; break; }
    got += (size_t)r;
  }
  buf_.resize(old + got);
  win_ = buf_.data(); win_len_ = buf_.size();
  return got > 0;
}

// One record at pos_.  Lines are found with memchr; nothing is copied here: the sequence lines become pieces.
int read_stream::scan_record(read_batch& b, uint64_t& nbases) {
  const char* w = win_;
  const size_t end = win_len_;
  size_t p = pos_;
  auto line_end = [&](size_t from, size_t& nl, size_t& len) -> bool {      // false: the window ends before the line does
    const char* q = from < end ? (const char*)memchr(w + from, '\n', end - from) : nullptr;
    if(!q) { if(!eof_) return false; nl = end; }                            // the last line may lack its terminator
    else nl = (size_t)(q - w);
    len = nl - from;
    if(len && w[from + len - 1] == '\r') --len;
    return true;
  };
  size_t nl, len;
  // header: skip empty lines
  while(true) {
    if(p >= end) return eof_ ? -1 : 0;
    if(!line_end(p, nl, len)) return 0;
    if(len) break;
    p = std::min(end, nl + 1);
  }
  const char c = w[p];
  if(c != '>' && c != '@') throw std::runtime_error("Unsupported format");
  if(!kind_) kind_ = c;
  const size_t hb = p + 1, he = p + len;
  size_t ws = hb;
  while(ws < he && !(w[ws] == ' ' || (w[ws] >= '\t' && w[ws] <= '\r'))) ++ws;
  p = std::min(end, nl + 1);
  const size_t first_piece = pieces_.size();
  uint64_t rlen = 0;
  if(c == '>') {
    while(true) {
      if(p >= end) { if(!eof_) { pieces_.resize(first_piece); return 0; } break; }
      if(w[p] == '>') break;
      if(!line_end(p, nl, len)) { pieces_.resize(first_piece); return 0; }
      if(len) { pieces_.push_back(piece{ (uint64_t)p, (uint32_t)len, nbases + rlen }); rlen += len; }
      p = std::min(end, nl + 1);
    }
  } else {
    bool plus = false;
    while(true) {                              // sequence lines up to the '+' line
      if(p >= end) { if(!eof_) { pieces_.resize(first_piece); return 0; } break; }
      if(!line_end(p, nl, len)) { pieces_.resize(first_piece); return 0; }
      const size_t at = p;
      p = std::min(end, nl + 1);
      if(len && w[at] == '+') { plus = true; break; }
      if(len) { pieces_.push_back(piece{ (uint64_t)at, (uint32_t)len, nbases + rlen }); rlen += len; }
    }
    uint64_t q = 0;
    while(plus && q < rlen) {                  // quality lines: as many characters as there were bases
      if(p >= end) { if(!eof_) { pieces_.resize(first_piece); return 0; } break; }
      if(!line_end(p, nl, len)) { pieces_.resize(first_piece); return 0; }
      q += len;
      p = std::min(end, nl + 1);
    }
  }
  b.name.emplace_back(w + hb, ws - hb);
  nbases += rlen;
  b.start.push_back(b.start.back() + rlen);
  pos_ = p;
  return 1;
}

// A mapped FASTA file: the records of the next 64 MB are found by all threads at once.  Thread t starts at the first
// record start ('>' at the beginning of a line) at or after its share of the stretch and stops at the next thread's, so
// every record is scanned by exactly one thread, whole; the per-thread lists are concatenated in file order.  One
// thread walking the file with memchr manages ~2 GB/s, which is what bounded the command-line tool (0.32 of its 0.38 s
// on 0.6 GB of reads).  The semantics are scan_record's: name up to the first white space, '\r' dropped, empty lines
// ignored, a sequence ends at the next '>' that starts a line.
bool read_stream::prescan() {
  pre_.clear(); pre_pieces_.clear(); pre_next_ = 0;
  if(!map_ || threads_ < 2 || pos_ >= win_len_ || win_[pos_] != '>' || kind_ == '@') return false;
  const char* w = win_;
  const size_t end = win_len_, A = pos_, B = std::min(end, A + ((size_t)64 << 20));
  const unsigned T = std::max(1u, std::min<unsigned>(threads_, (unsigned)((B - A) >> 20) + 1));
  auto find_start = [&](size_t p) -> size_t {
    while(p < end) {
      const char* q = (const char*)memchr(w + p, '>', end - p);
      if(!q) return end;
      const size_t at = (size_t)(q - w);
      if(at == 0 || w[at - 1] == '\n') return at;
      p = at + 1;
    }
    return end;
  };
  std::vector<size_t> s(T + 1, end);
  std::vector<std::vector<prerec>> recs(T);
  std::vector<std::vector<piece>> pcs(T);
  auto locate = [&](unsigned t) { s[t] = t == 0 ? A : find_start(A + (B - A) / T * t); };
  auto scan = [&](unsigned t) {
    size_t p = s[t];
    const size_t stop = s[t + 1];
    auto line_end = [&](size_t from, size_t& nl, size_t& len) {
      const char* q = from < end ? (const char*)memchr(w + from, '\n', end - from) : nullptr;
      nl = q ? (size_t)(q - w) : end;
      len = nl - from;
      if(len && w[from + len - 1] == '\r') --len;
    };
    while(p < stop) {
      size_t nl, len;
      line_end(p, nl, len);                            // the header line: w[p] == '>'
      const size_t hb = p + 1, he = p + len;
      size_t ws = hb;
      while(ws < he && !(w[ws] == ' ' || (w[ws] >= '\t' && w[ws] <= '\r'))) ++ws;
      prerec r;
      r.name_b = hb; r.name_len = (uint32_t)(ws - hb); r.first_piece = pcs[t].size(); r.npieces = 0; r.len = 0;
      p = std::min(end, nl + 1);
      while(p < end && w[p] != '>') {
        line_end(p, nl, len);
        if(len) { pcs[t].push_back(piece{ (uint64_t)p, (uint32_t)len, 0 }); ++r.npieces; r.len += len; }
        p = std::min(end, nl + 1);
      }
      r.end_pos = p;
      recs[t].push_back(r);
    }
  };
  auto run = [&](const std::function<void(unsigned)>& f) {
    std::vector<std::thread> th;
    for(unsigned t = 1; t < T; ++t) th.emplace_back(f, t);
    f(0);
    for(auto& x : th) x.join();
  };
  run(locate);
  s[T] = find_start(B);
  for(unsigned t = 1; t <= T; ++t) if(s[t] < s[t - 1]) s[t] = s[t - 1];
  run(scan);
  for(unsigned t = 0; t < T; ++t) {
    const uint64_t shift = pre_pieces_.size();
    for(prerec r : recs[t]) { r.first_piece += shift; pre_.push_back(r); }
    pre_pieces_.insert(pre_pieces_.end(), pcs[t].begin(), pcs[t].end());
  }
  if(!pre_.empty() && !kind_) kind_ = '>';
  return !pre_.empty();
}

bool read_stream::next_batch(read_batch& b, uint64_t max_bases, uint32_t max_reads, bool pack) {
  if(b.start.empty()) b.start.push_back(0);
  const uint64_t base0 = b.bases.size();
  // ---- serial: find the records --------------------------------------------------------------------
  // pieces of one batch may come from several files; each group is copied before its window goes away
  uint64_t nbases = base0;
  bool any = false;
  auto flush_pieces = [&]() {
    if(pieces_.empty()) { b.bases.resize(nbases); return; }
    b.bases.resize(nbases);
    char* dst = &b.bases[0];
    const char* w = win_;
    const unsigned nt = std::max(1u, std::min<unsigned>(threads_, (unsigned)(pieces_.size() / 64 + 1)));
    auto work = [&](unsigned t) {
      const size_t lo = pieces_.size() * t / nt, hi = pieces_.size() * (t + 1) / nt;
      for(size_t i = lo; i < hi; ++i) memcpy(dst + pieces_[i].dst, w + pieces_[i].src, pieces_[i].len);
    };
    if(nt == 1) work(0);
    else {
      std::vector<std::thread> th;
      for(unsigned t = 0; t < nt; ++t) th.emplace_back(work, t);
      for(auto& x : th) x.join();
    }
    pieces_.clear();
  };
  while(nbases - b.start[0] < max_bases && b.nreads() < max_reads) {
    if(!open_) {
      if(!open_next()) break;
    }
    if(!map_ && pieces_.empty() && pos_ > 0 && pos_ == win_len_) { buf_.clear(); win_ = nullptr; win_len_ = 0; pos_ = 0; }
    if(map_ && threads_ > 1 && (pre_next_ < pre_.size() || prescan())) {     // a record the threads found ahead
      const prerec& r = pre_[pre_next_++];
      b.name.emplace_back(win_ + r.name_b, r.name_len);
      uint64_t rlen = 0;
      for(uint32_t i = 0; i < r.npieces; ++i) {
        const piece& pc = pre_pieces_[r.first_piece + i];
        pieces_.push_back(piece{ pc.src, pc.len, nbases + rlen });
        rlen += pc.len;
      }
      nbases += rlen;
      b.start.push_back(b.start.back() + rlen);
      pos_ = r.end_pos;
      any = true;
      continue;
    }
    const int rc = scan_record(b, nbases);
    if(rc == 1) { any = true; continue; }
    if(rc == 0) {                               // stream mode: the record continues behind the window
      if(pieces_.empty() && pos_ > 0) {         // nothing points into the consumed part: drop it
        buf_.erase(buf_.begin(), buf_.begin() + (ptrdiff_t)pos_);
        pos_ = 0; win_ = buf_.data(); win_len_ = buf_.size();
      }
      refill();
      continue;
    }
    flush_pieces();                             // end of this file
    close_current();
  }
  flush_pieces();
  // in stream mode the consumed prefix is dropped now that no piece points into it
  if(open_ && !map_ && pos_ > 0) {
    buf_.erase(buf_.begin(), buf_.begin() + (ptrdiff_t)pos_);
    pos_ = 0; win_ = buf_.data(); win_len_ = buf_.size();
  }
  // ---- parallel: pack --------------------------------------------------------------------------------
  if(pack && any) {
    const uint64_t n = b.bases.size();
    b.size_packed(mr_packed_code_words(n), mr_packed_mask_words(n));
    const uint64_t mwords = b.nmask.size();
    const unsigned nt = std::max(1u, std::min<unsigned>(threads_, (unsigned)(mwords / 4096 + 1)));
    auto work = [&](unsigned t) {
      if(nt > 1) background_thread();
      const uint64_t lo = mwords * t / nt, hi = mwords * (t + 1) / nt;
      mr_pack_reads_range(b.bases.data(), n, lo, hi - lo, b.codes.data(), b.nmask.data());
    };
    if(nt == 1) work(0);
    else {
      std::vector<std::thread> th;
      for(unsigned t = 0; t < nt; ++t) th.emplace_back(work, t);
      for(auto& x : th) x.join();
    }
  }
  return any;
}

// ================================================================================================
// mega-reads from the device's graph rows
// ================================================================================================
namespace {
// the number formatters of a mega-read line (overlap_graph.cc:285-290), shared with the device's printer
using mrfmt::fmt_int;
using mrfmt::fmt_uint;
using mrfmt::fmt_fixed;

struct mega_read {
  int    start_node, end_node, start_unitig, start_offset, end_offset, nb_unitigs;
  double imp_s, imp_e, tiling_start, tiling_end, density;
};
struct span { double lo, up; };

// joining interval set of [lo, up) pieces: boost::icl::interval_set<double> as used by tile_greedy
struct joined_set {
  std::vector<span> v, nv;                     // nv: scratch of add(), kept so that a read's tiling does not allocate per piece
  void clear() { v.clear(); }
  bool overlaps_at_least(const span& x, double limit) const {
    for(const span& y : v) {
      const double lo = std::max(y.lo, x.lo), up = std::min(y.up, x.up);
      if(lo < up && up - lo >= limit) return true;
    }
    return false;
  }
  void add(span x) {
    if(!(x.lo < x.up)) return;
    nv.clear();
    bool placed = false;
    for(const span& y : v) {
      if(y.up < x.lo) nv.push_back(y);
      else if(x.up < y.lo) { if(!placed) { nv.push_back(x); placed = true; } nv.push_back(y); }
      else { x.lo = std::min(x.lo, y.lo); x.up = std::max(x.up, y.up); }
    }
    if(!placed) nv.push_back(x);
    v.swap(nv);
  }
};
} // namespace

uint64_t selftest_fixed_format(uint64_t samples, uint64_t seed) {
  uint64_t state = seed * 0x9e3779b97f4a7c15ULL + 1, bad = 0;
  auto next = [&]() { state ^= state << 13; state ^= state >> 7; state ^= state << 17; return state; };
  char a[80], b[80];
  auto check = [&](double x) {
    for(int d = 2; d <= 4; d += 2) {
      const int n = fmt_fixed(a, x, d);
      a[n] = 0;
      snprintf(b, sizeof b, "%.*f", d, x);
      bad += strcmp(a, b) != 0;
    }
  };
  const double fixed[] = { 0.0, 0.125, 0.375, 2.675, 1.005, 0.005, 0.015, 0.025, 0.00005, 0.00015, 1e-13, 0.5, 1.5, 2.5, 0.045,
                           99999.995, 12345.675, 1e10, 9.99999e10, 1e11, 3.14159, 0.999999, 0.995, 0.99995, 4.35, 4.345, 1e-300, 5e-324 };
  for(double x : fixed) { check(x); check(-x); }
  for(uint64_t i = 0; i < samples; ++i) {
    double x;
    const uint64_t r = next();
    switch(i & 7) {
    case 0: x = (double)(r % 2000000) / 100.0; break;
    case 1: x = (double)(r % 200000000) / 10000.0; break;
    case 2: x = (double)(r % 4000001) / 200.0; break;            // decimal half-way points
    case 3: x = (double)(r % 40000001) / 20000.0; break;
    case 4: x = std::ldexp((double)(r >> 11), -53) * 20000.0; break;
    case 5: x = std::ldexp((double)(r >> 11), -53); break;
    case 6: x = (double)(r % 1000000) / 1024.0; break;           // binary fractions: exact ties
    default: x = std::ldexp((double)(r >> 11), -53 + (int)(next() % 40) - 10); break;
    }
    check(next() & 1 ? -x : x);
  }
  return bad;
}

namespace {
// --dot, first half of a read's graph: header, node tooltips in node order, and the overlap edges in the order
// overlap_graph::traverse finds them (overlap_graph.cc:7-59, with the edge test redone on the host)
void dot_open_read(const mr_result_view& v, const read_batch& batch, uint32_t r, const super_reads& sr, const unitigs& u,
                   const graph_options& o, const dot_state& ds, text_buf& dot) {
  char buf[160];
  const uint64_t b = v.read_coords[r];
  const int n = (int)(v.read_coords[r + 1] - b);
  dot += "digraph \""; dot += batch.name[r]; dot += "\" {\nnode [fontsize=\"10\"];\n";
  if(n == 0) return;
  const double rl = (double)(batch.start[r + 1] - batch.start[r]), K = o.k_len;
  std::vector<double> imp_s(n), imp_e(n);
  std::vector<int> order(n);
  for(int i = 0; i < n; ++i) {
    const uint64_t row = b + i;
    imp_s[i] = v.stretch[row] + v.offset[row];
    const double t = v.stretch[row] * (double)v.ql[row];
    imp_e[i] = t + v.offset[row];
    order[i] = i;
  }
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return imp_s[x] < imp_s[y] || (imp_s[x] == imp_s[y] && imp_e[x] < imp_e[y]); });
  for(int a = 0; a < n; ++a) {
    snprintf(buf, sizeof buf, "n%d[tooltip=\"", order[a]);
    dot += buf; dot += sr.row_name(v.sr[b + order[a]], v.use_bwd[b + order[a]]); dot += "\"];\n";
  }
  auto path_len = [&](uint64_t row) { return sr.path_len(v.sr[row]); };
  auto path_at = [&](uint64_t row, uint32_t t) { return sr.path_at(v.sr[row], v.use_bwd[row], t); };
  for(int a = 0; a < n; ++a) {
    const int ii = order[a];
    const uint64_t ri = b + ii;
    if(imp_e[ii] >= rl) continue;
    const uint32_t ln = path_len(ri);
    for(int bb = a + 1; bb < n; ++bb) {
      const int jj = order[bb];
      const uint64_t rj = b + jj;
      if(imp_s[jj] <= 1 || imp_e[ii] > imp_e[jj] + 31) continue;
      const double position_len = imp_e[ii] - imp_s[jj];
      const double error1 = v.avg_err[ri] + v.avg_err[rj];
      const double error = ds.errors * error1;
      const double ppl = position_len * o.overlap_play;
      if(ppl + error < K) break;
      const uint32_t rn = path_len(rj);
      int nb_u = 0;                                       // super_read_name::overlap (super_read_name.cc:49-72)
      if(ln >= 2 && rn >= 2) {
        for(uint32_t i = (uint32_t)std::max<int64_t>(1, (int64_t)ln - (int64_t)rn + 1); i < ln && !nb_u; ++i) {
          if(path_at(ri, i) != path_at(rj, 0)) continue;
          uint32_t j = i + 1;
          while(j < ln && path_at(ri, j) == path_at(rj, j - i)) ++j;
          if(j == ln) nb_u = (int)(ln - i);
        }
      }
      if(!nb_u) continue;
      bool same = ln == rn;
      for(uint32_t t = 0; same && t < ln; ++t) same = path_at(ri, t) == path_at(rj, t);
      if(same) continue;
      int u_len = 0, common = 0;
      const uint32_t ilen = v.info_len[rj];
      const int32_t* info = (ds.bases ? v.bases_info : v.kmers_info) + v.info_off[rj];
      for(int t = 0; t < nb_u; ++t) {
        const uint32_t id = path_at(rj, (uint32_t)t) >> 1;
        u_len += id < u.len.size() ? u.len[id] : 0;
        if((uint32_t)(2 * t) < ilen) common += info[2 * t];
        if(t > 0 && (uint32_t)(2 * t - 1) < ilen) common -= info[2 * t - 1];
      }
      u_len -= (nb_u - 1) * ((int)o.k_len - 1);
      const double t1 = o.overlap_play * position_len, t2 = o.overlap_play * ((double)u_len + error);
      if((double)u_len > t1 + error || position_len > t2) continue;
      snprintf(buf, sizeof buf, "n%d -> n%d [tooltip=\"...\", label=\"%d\"];\n", ii, jj, common);
      dot += buf;
    }
  }
}
} // namespace

void format_mega_reads(const mr_result_view& v, const read_batch& batch, uint32_t r0, uint32_t r1,
                       const super_reads& sr, const unitigs& u, const graph_options& o, text_buf& out,
                       text_buf* dot, dot_state* ds) {
  const double K = o.k_len;
  std::vector<mega_read> mrs;
  std::vector<int> sort_tiling, tiled;
  std::vector<uint32_t> path;
  std::vector<double> weights;
  struct seq_piece { const char* p; size_t n; };
  std::vector<seq_piece> pieces;
  std::vector<int> comp_slot, comp_root;
  std::vector<mega_read> comp_mr;
  joined_set covered;
  std::vector<span> placed;
  char buf[4 * mrfmt::kFixedMax];
  // ids come from super-read names, lengths from the -l/-u table: the libraries refuse a table that
  // does not cover the names (mr_align_batch, mr_graph_batch), this keeps a stray id from reading
  // past the table all the same
  auto ulen_of = [&](uint32_t id) -> int { return id < u.len.size() ? u.len[id] : 0; };
  for(uint32_t r = r0; r < r1; ++r) {
    const uint64_t b = v.read_coords[r];
    const int n = (int)(v.read_coords[r + 1] - b);
    if(dot) dot_open_read(v, batch, r, sr, u, o, *ds, *dot);      // (the reference opens a graph for every read, also one without rows)
    if(n == 0) continue;
    const double pb_size = (double)(batch.start[r + 1] - batch.start[r]);
    auto row_unitig_id = [&](uint64_t row, uint32_t t) -> uint32_t {
      const uint32_t s = v.sr[row];
      return t < sr.path_len(s) ? (sr.path_at(s, v.use_bwd[row], t) >> 1) : 0x7fffffffu;
    };

    // mega_reads_per_comp (overlap_graph.cc:116-161): the best mega-read of every component, components in increasing
    // root order (the reference keeps them in a std::map keyed by the root; a root is a node number below n, so a table
    // of slots does the same without a tree node per component)
    comp_slot.assign((size_t)n, -1);
    comp_mr.clear(); comp_root.clear();
    for(int i = 0; i < n; ++i) {
      const uint64_t row = b + i;
      mega_read mr;
      mr.start_node = v.lstart[row] == -1 ? i : v.lstart[row];
      mr.end_node = i;
      const uint64_t srow = b + mr.start_node;
      mr.start_unitig = 0;
      mr.nb_unitigs = v.lunitigs[row];
      mr.imp_s = v.stretch[srow] + v.offset[srow];
      { const double t = v.stretch[row] * (double)v.ql[row]; mr.imp_e = t + v.offset[row]; }
      mr.tiling_start = v.rs[srow];
      mr.tiling_end = v.re[row];
      mr.start_offset = mr.end_offset = 0;
      if(o.trim != 0) {                                   // trim_match (overlap_graph.cc:78-114)
        const double node_imp_s = v.stretch[srow] + v.offset[srow];
        if(node_imp_s < 1) {
          const int32_t* ki = v.kmers_info + v.info_off[srow];
          const int ilen = (int)v.info_len[srow];
          int offset = 0, su = 0;
          for(su = 0; su < ilen; su += 2) {
            if(ki[su]) break;
            offset += ulen_of(row_unitig_id(srow, su / 2));
          }
          su /= 2;
          mr.start_unitig = su;
          mr.nb_unitigs -= su;
          offset -= ((int)o.k_len - 1) * su;
          mr.start_offset = offset;
          { const double t = v.stretch[srow] * (double)(offset + 1); mr.imp_s = t + v.offset[srow]; }
        }
        const double node_imp_e = mr.imp_e;
        if(node_imp_e > (double)v.ql[row]) {
          const int32_t* ki = v.kmers_info + v.info_off[row];
          const int ilen = (int)v.info_len[row];
          int offset = 0, eu;
          for(eu = ilen - 1; eu >= 0; eu -= 2) {
            if(ki[eu]) break;
            offset += ulen_of(row_unitig_id(row, eu / 2));
          }
          eu /= 2;
          const int removed = ilen / 2 - eu;
          mr.nb_unitigs -= removed;
          offset -= ((int)o.k_len - 1) * removed;
          mr.end_offset = offset;
          { const double t = v.stretch[row] * (double)((int64_t)v.ql[row] - offset); mr.imp_e = t + v.offset[row]; }
        }
      }
      const double len = std::min(pb_size + 0.5, mr.tiling_end) - std::max(0.5, mr.tiling_start);
      mr.density = (double)v.lpath[row] / len;
      if(dot) {                                            // node label (overlap_graph.cc:133-146)
        char db[400];
        const double node_s = v.stretch[row] + v.offset[row];
        const double node_e = v.stretch[row] * (double)v.ql[row] + v.offset[row];
        const int prec = ds->first_node ? 6 : 2;           // the stream's precision: 6 until the first density sets it to 2
        ds->first_node = false;
        snprintf(db, sizeof db, "n%d [label=\"%d L%u #%d\\nP(%d,%d) S(%d,%d)\\nI(%.*f,%.*f)\\nLP #%d L%.1f d%.2f\"%s];\n", i, i, v.ql[row],
                 v.nb_mers[row], v.rs[row], v.re[row], v.qs[row], v.qe[row], prec, node_s, prec, node_e, v.lpath[row], len, mr.density,
                 v.start_node[row] ? ", color=\"blue\"" : (v.end_node[row] ? ", color=\"green\"" : ""));
        *dot += db;
      }
      if(!v.end_node[row] || mr.density < o.density || (mr.tiling_end - mr.tiling_start) < o.min_length) continue;
      const int root = v.component[row];
      if(root < 0 || root >= n) throw std::out_of_range("component root outside the read's rows");
      const int slot = comp_slot[(size_t)root];
      if(slot < 0) { comp_slot[(size_t)root] = (int)comp_mr.size(); comp_mr.push_back(mr); comp_root.push_back(root); }
      else {
        mega_read& cur = comp_mr[(size_t)slot];
        const int olpath = v.lpath[b + cur.end_node];
        if(v.lpath[row] > olpath || (v.lpath[row] == olpath && mr.density > cur.density)) cur = mr;
      }
    }
    if(comp_mr.empty()) continue;
    mrs.clear(); sort_tiling.clear(); tiled.clear();
    for(int root = 0; root < n; ++root)
      if(comp_slot[(size_t)root] >= 0) { sort_tiling.push_back((int)mrs.size()); mrs.push_back(comp_mr[(size_t)comp_slot[(size_t)root]]); }
    auto lpath_of = [&](int m) { return v.lpath[b + mrs[m].end_node]; };
    auto by_pos = [&](int i, int j) {
      return mrs[i].imp_s < mrs[j].imp_s || (mrs[i].imp_s == mrs[j].imp_s && mrs[i].imp_e < mrs[j].imp_e);
    };
    auto greedy = [&]() {                                  // tile_greedy (overlap_graph.cc:165-197)
      covered.clear();
      placed.clear();
      for(const int m : sort_tiling) {
        const span pos = { mrs[m].tiling_start, mrs[m].tiling_end };
        const double plen = pos.lo < pos.up ? pos.up - pos.lo : 0.0;
        const double max_overlap = std::max(K * o.overlap_play, plen * (o.overlap_play - 0.9));
        if(covered.overlaps_at_least(pos, max_overlap)) continue;
        bool contained = false;
        for(const span& p : placed)
          if(!(pos.lo < pos.up) || (p.lo <= pos.lo && pos.up <= p.up)) { contained = true; break; }
        if(contained) continue;
        covered.add(pos);
        placed.push_back(pos);
        tiled.push_back(m);
      }
    };
    // the std::sort calls below are the reference's own (same comparator, same input order), so
    // even their unspecified order on ties is reproduced
    switch(o.tiling) {
    case 1:
      std::sort(sort_tiling.begin(), sort_tiling.end(), [&](int i, int j) { return lpath_of(j) < lpath_of(i); });
      greedy();
      std::sort(tiled.begin(), tiled.end(), by_pos);
      break;
    case 3:
      weights.assign(mrs.size(), 0.0);
      for(const int i : sort_tiling) {
        const double d2 = mrs[i].density * mrs[i].density;
        weights[i] = d2 * (double)(v.re[b + mrs[i].end_node] - v.rs[b + mrs[i].start_node] + 1);
      }
      std::sort(sort_tiling.begin(), sort_tiling.end(), [&](int i, int j) { return weights[j] < weights[i]; });
      greedy();
      std::sort(tiled.begin(), tiled.end(), by_pos);
      break;
    case 2: {                                              // tile_maximal (overlap_graph.cc:212-252)
      std::sort(sort_tiling.begin(), sort_tiling.end(), [&](int i, int j) { return mrs[i].tiling_end < mrs[j].tiling_end; });
      struct tinfo { int score; double pos; int node, previous, length; };
      std::vector<tinfo> info;
      auto it = sort_tiling.begin();
      info.push_back({ lpath_of(*it), mrs[*it].tiling_end, *it, -1, 1 });
      for(++it; it != sort_tiling.end(); ++it) {
        const double lstart = mrs[*it].tiling_start;
        const double key = std::min(lstart + K * o.overlap_play, mrs[*it].tiling_end);
        int i = (int)(std::upper_bound(info.begin(), info.end(), key, [](double x, const tinfo& y) { return x < y.pos; }) - info.begin()) - 1;
        while(i >= 0 && mrs[info[i].node].tiling_start >= lstart) i = info[i].previous;
        const int nscore = (i >= 0 ? info[i].score : 0) + lpath_of(*it);
        if(nscore > info.back().score) info.push_back({ nscore, mrs[*it].tiling_end, *it, i, (i >= 0 ? info[i].length : 0) + 1 });
      }
      tiled.resize(info.back().length);
      int ptr = (int)info.size() - 1;
      for(auto rit = tiled.rbegin(); rit != tiled.rend(); ++rit) { *rit = info[ptr].node; ptr = info[ptr].previous; }
      std::sort(tiled.begin(), tiled.end(), by_pos);
      break;
    }
    default: break;
    }

    // print_mega_reads (overlap_graph.hpp:253-262, overlap_graph.cc:254-299)
    out += '>'; out += batch.name[r]; out += '\n';
    const std::vector<int>& final_order = tiled.empty() ? sort_tiling : tiled;
    for(const int cmr : final_order) {
      const mega_read& mr = mrs[cmr];
      const uint64_t erow = b + mr.end_node, srow = b + mr.start_node;
      path.assign((size_t)std::max(0, v.lunitigs[erow]), 0u);
      auto prepend = [&](size_t offset, uint64_t row, size_t first, size_t last) -> size_t {
        const uint32_t s = v.sr[row];
        const size_t sz = sr.path_len(s);
        if(first > last || first >= sz) return offset;
        const size_t to_copy = std::min(last, sz - 1) - first + 1;
        if(to_copy > offset) return offset;
        for(size_t t = 0; t < to_copy; ++t) path[offset - to_copy + t] = sr.path_at(s, v.use_bwd[row], (uint32_t)(first + t));
        return offset - to_copy;
      };
      size_t offset = prepend(path.size(), erow, 0, (size_t)sr.path_len(v.sr[erow]) - 1);
      int node_j = mr.end_node, node_i = v.lprev[erow];
      while(node_i >= 0) {
        const uint64_t irow = b + node_i, jrow = b + node_j;
        const size_t overlap = (size_t)v.lunitigs[irow] + sr.path_len(v.sr[jrow]) - (size_t)v.lunitigs[jrow];
        const size_t end = (size_t)sr.path_len(v.sr[irow]) - 1 - overlap;
        offset = prepend(offset, irow, 0, end);
        if(dot) { char db[80]; snprintf(db, sizeof db, "n%d -> n%d [color=\"red\"];\n", node_i, node_j); *dot += db; }
        node_j = node_i;
        node_i = v.lprev[irow];
      }
      auto path_id = [&](int i) -> uint32_t { return (size_t)i < path.size() ? (path[i] >> 1) : 0x7fffffffu; };
      int sr_len = 0;
      for(int i = mr.start_unitig; i < mr.start_unitig + mr.nb_unitigs; ++i) sr_len += ulen_of(path_id(i));
      sr_len -= (mr.nb_unitigs - 1) * ((int)o.k_len - 1);
      const uint64_t qe_out = (uint64_t)(int64_t)(sr_len + mr.end_offset) - ((uint64_t)v.ql[erow] - (uint64_t)(int64_t)v.qe[erow]);
      // "%.2f %.2f %d %d %d %llu %d %.4f " (overlap_graph.cc:285-290), then "<id><F|R>" joined by '_', " sr_len"
      char* w = buf;
      w += fmt_fixed(w, mr.imp_s, 2); *w++ = ' ';
      w += fmt_fixed(w, mr.imp_e, 2); *w++ = ' ';
      w += fmt_int(w, v.rs[srow]); *w++ = ' ';
      w += fmt_int(w, v.re[erow]); *w++ = ' ';
      w += fmt_int(w, v.qs[srow] - mr.start_offset); *w++ = ' ';
      w += fmt_uint(w, qe_out); *w++ = ' ';
      w += fmt_int(w, v.lpath[erow]); *w++ = ' ';
      w += fmt_fixed(w, mr.density, 4); *w++ = ' ';
      for(size_t t = 0; t < path.size(); ++t) {
        if(w - buf > (ptrdiff_t)sizeof(buf) - 32) { out.append(buf, (size_t)(w - buf)); w = buf; }
        if(t) *w++ = '_';
        w += fmt_uint(w, path[t] >> 1);
        *w++ = (path[t] & 1) ? 'R' : 'F';
      }
      *w++ = ' ';
      w += fmt_int(w, sr_len);
      if(u.has_sequences()) {                             // super_read_name::print_sequence (super_read_name.cc:123-132)
        *w++ = ' ';
        out.append(buf, (size_t)(w - buf)); w = buf;
        const size_t pb = std::min((size_t)mr.start_unitig, path.size());
        const size_t pe = std::min((size_t)(mr.start_unitig + mr.nb_unitigs), path.size());
        const size_t nu = u.len.size();
        // The sequence is a splice of ~400-byte pieces scattered over the unitig arena (tens of MB: cache misses).
        // All pieces of the line are located first, their first lines requested as they are found, and only then
        // copied -- into space taken once for the whole line -- so the misses overlap instead of queueing one per piece.
        pieces.clear();
        size_t total = 0;
        for(size_t i = pb; i < pe; ++i) {
          const uint32_t id = path[i] >> 1;
          if(id >= nu) throw std::out_of_range("unitig id of a super-read name is not in the -u file");   // vector::at in the reference
          const size_t sl = (size_t)u.len[id], skip = i == pb ? 0 : (size_t)o.k_len - 1;
          if(skip >= sl) continue;
          const char* src = u.sequence(id, path[i] & 1) + skip;
          __builtin_prefetch(src); __builtin_prefetch(src + 64); __builtin_prefetch(src + 128); __builtin_prefetch(src + 192);
          pieces.push_back(seq_piece{ src, sl - skip });
          total += sl - skip;
        }
        char* dst = out.grab(total);
        for(const seq_piece& pc : pieces) { memcpy(dst, pc.p, pc.n); dst += pc.n; }
      }
      *w++ = '\n';
      out.append(buf, (size_t)(w - buf));
    }
    if(dot) *dot += "}\n";                       // only reads with mega-reads get their graph closed (overlap_graph.hpp:258-259)
  }
}

// default ostream formatting of a double: "%g" with 6 significant digits (jf_aligner.cc:58)
void format_coords(const mr_result_view& v, const read_batch& batch, uint32_t r0, uint32_t r1, const super_reads& sr,
                   bool compact, bool zero_skip, text_buf& out) {
  char buf[512];
  for(uint32_t r = r0; r < r1; ++r) {
    const uint64_t b = v.read_coords[r], e = v.read_coords[r + 1];
    if(b == e && zero_skip) continue;
    const uint64_t pb_size = batch.start[r + 1] - batch.start[r];
    if(compact) {
      snprintf(buf, sizeof(buf), ">%llu ", (unsigned long long)(e - b));
      out += buf; out += batch.name[r]; out += '\n';
    }
    for(uint64_t row = b; row < e; ++row) {
      if(!compact) { out += batch.name[r]; out += ' '; }
      snprintf(buf, sizeof(buf), "%d %d %d %d %d %u %u %u %u %llu %u %g %g %g ", v.rs[row], v.re[row], v.qs[row], v.qe[row],
               v.nb_mers[row], v.pb_cons[row], v.sr_cons[row], v.pb_cover[row], v.sr_cover[row],
               (unsigned long long)pb_size, v.ql[row], v.stretch[row], v.offset[row], v.avg_err[row]);
      out += buf;
      out += sr.row_name(v.sr[row], v.use_bwd[row]);
      const int32_t* ki = v.kmers_info + v.info_off[row];
      const int32_t* bi = v.bases_info + v.info_off[row];
      for(uint32_t t = 0; t < v.info_len[row]; ++t) {
        snprintf(buf, sizeof(buf), " %d:%d", ki[t], bi[t]);
        out += buf;
      }
      out += '\n';
    }
  }
}

void format_details(const mr_result* r, const read_batch& batch, const super_reads& sr, text_buf& out) {
  uint64_t ng = 0, no = 0, nl = 0;
  const int64_t* groups = nullptr; const int32_t* offsets = nullptr; const uint32_t* lis = nullptr;
  if(mr_result_taps(r, &ng, &groups, &no, &offsets, &nl, &lis) != MR_OK) return;
  char buf[64];
  uint64_t off = 0, li = 0;
  for(uint64_t g = 0; g < ng; ++g) {
    const int64_t* row = groups + 6 * g;
    const uint64_t nf = row[2], nb = row[3], lf = row[4], lb = row[5];
    const int32_t* fwd = offsets + 2 * off; const int32_t* bwd = fwd + 2 * nf;
    const uint32_t* lis_f = lis + li; const uint32_t* lis_b = lis_f + lf;
    out += batch.name[row[0]]; out += ' '; out += sr.name[row[1]];
    const bool fwd_align = lf > lb;                      // strict, unlike compute_coords_info
    const uint32_t* lit = fwd_align ? lis_f : lis_b;
    const uint32_t* lend = lit + (fwd_align ? lf : lb);
    uint64_t fi = 0, bi = 0;
    while(fi < nf || bi < nb) {
      int32_t pb = 0, so = 0; bool in_lis = false, took = false;
      if(fi < nf && (bi == nb || fwd[2 * fi] <= bwd[2 * bi])) {
        pb = fwd[2 * fi]; so = fwd[2 * fi + 1];
        in_lis = fwd_align && lit < lend && *lit == fi;
        ++fi; took = true;
      } else if(bi < nb && (fi == nf || bwd[2 * bi] < fwd[2 * fi])) {
        pb = bwd[2 * bi]; so = bwd[2 * bi + 1];
        in_lis = !fwd_align && lit < lend && *lit == bi;
        ++bi; took = true;
      }
      if(!took) break;
      snprintf(buf, sizeof(buf), in_lis ? " [%d:%d]" : " %d:%d", pb, so);
      out += buf;
      if(in_lis) ++lit;
    }
    out += '\n';
    off += nf + nb; li += lf + lb;
  }
}

// ================================================================================================
// compact coords files
// ================================================================================================
void coords_batch::clear() {
  reads.clear(); read_len.clear();
  paths = super_reads();
  paths.unitig_off.push_back(0);
  read_coords.assign(1, 0); info_off.clear();
  rs.clear(); re.clear(); qs.clear(); qe.clear(); nb_mers.clear(); kmers_info.clear(); bases_info.clear();
  pb_cons.clear(); sr_cons.clear(); pb_cover.clear(); sr_cover.clear(); ql.clear(); sr.clear(); info_len.clear();
  rn.clear(); use_bwd.clear(); stretch.clear(); offset.clear(); avg_err.clear();
}

mr_result_view coords_batch::view() const {
  mr_result_view v;
  memset(&v, 0, sizeof v);
  v.nreads = reads.nreads(); v.ncoords = rs.size(); v.read_coords = read_coords.data();
  v.rs = rs.data(); v.re = re.data(); v.qs = qs.data(); v.qe = qe.data(); v.nb_mers = nb_mers.data();
  v.pb_cons = pb_cons.data(); v.sr_cons = sr_cons.data(); v.pb_cover = pb_cover.data(); v.sr_cover = sr_cover.data();
  v.ql = ql.data(); v.sr = sr.data(); v.rn = rn.data(); v.use_bwd = use_bwd.data();
  v.stretch = stretch.data(); v.offset = offset.data(); v.avg_err = avg_err.data();
  v.info_off = info_off.data(); v.info_len = info_len.data();
  v.kmers_info = kmers_info.data(); v.bases_info = bases_info.data();
  return v;
}

coords_file::coords_file(const std::string& path) : f_(fopen(path.c_str(), "r")) {
  if(!f_) throw std::runtime_error("Failed to open coords file '" + path + "'");
}

bool coords_file::getline() {
  line_.clear();
  char buf[1 << 16];
  bool any = false;
  while(fgets(buf, sizeof buf, f_)) {
    any = true;
    const size_t len = strlen(buf);
    if(len && buf[len - 1] == '\n') { line_.append(buf, len - 1); return true; }
    line_.append(buf, len);
  }
  return any;
}

bool coords_file::next_batch(coords_batch& b, uint64_t max_rows) {
  b.clear();
  if(!started_) {                              // skip the column header: everything before the first '>' line
    started_ = true;
    while((pending_ = getline()) && (line_.empty() || line_[0] != '>')) { }
  }
  std::vector<uint32_t> upath;
  while(pending_ && b.rs.size() < max_rows) {
    if(line_.empty() || line_[0] != '>') throw std::runtime_error("Invalid input file. Line expected to match /^>/ but got: " + line_);
    char* end = nullptr;
    errno = 0;
    const long nb_lines = strtol(line_.c_str() + 1, &end, 10);
    if(nb_lines <= 0 || errno == ERANGE) throw std::runtime_error("Invalid input file. Expected number of lines but got: " + line_.substr(1));
    b.reads.name.push_back(*end ? std::string(end + 1) : std::string());
    uint32_t rl_first = 0;
    for(long j = 0; j < nb_lines; ++j) {
      if(!getline()) throw std::runtime_error("Invalid input file. File truncated");
      const char* p = line_.c_str();
      char* q = nullptr;
      auto integer = [&]() -> long { const long v = strtol(p, &q, 10); p = q; return v; };
      auto real = [&]() -> double { const double v = strtod(p, &q); p = q; return v; };
      b.rs.push_back((int32_t)integer()); b.re.push_back((int32_t)integer());
      b.qs.push_back((int32_t)integer()); b.qe.push_back((int32_t)integer());
      b.nb_mers.push_back((int32_t)integer());
      b.pb_cons.push_back((uint32_t)integer()); b.sr_cons.push_back((uint32_t)integer());
      b.pb_cover.push_back((uint32_t)integer()); b.sr_cover.push_back((uint32_t)integer());
      const uint32_t rl = (uint32_t)integer();
      if(j == 0) rl_first = rl;
      b.ql.push_back((uint32_t)integer());
      b.stretch.push_back(real()); b.offset.push_back(real()); b.avg_err.push_back(real());
      while(*p == ' ' || *p == '\t') ++p;
      const char* ne = p;
      while(*ne && *ne != ' ' && *ne != '\t') ++ne;
      b.paths.name.emplace_back(p, ne);
      parse_path(b.paths.name.back(), upath);
      b.paths.unitig_ids.insert(b.paths.unitig_ids.end(), upath.begin(), upath.end());
      b.paths.unitig_off.push_back(b.paths.unitig_ids.size());
      b.sr.push_back((uint32_t)(b.paths.name.size() - 1));
      b.rn.push_back(0); b.use_bwd.push_back(0);
      p = ne;
      b.info_off.push_back(b.kmers_info.size());
      uint32_t ninfo = 0;
      while(true) {                            // "mers:bases" pairs until something else
        const long m = strtol(p, &q, 10);
        if(q == p || *q != ':') break;
        const char* p2 = q + 1;
        const long bs = strtol(p2, &q, 10);
        if(q == p2) break;
        b.kmers_info.push_back((int32_t)m); b.bases_info.push_back((int32_t)bs);
        ++ninfo;
        p = q;
      }
      b.info_len.push_back(ninfo);
    }
    b.read_len.push_back(rl_first);
    b.reads.start.push_back(b.reads.start.back() + rl_first);
    b.read_coords.push_back(b.rs.size());
    pending_ = getline();
  }
  return b.reads.nreads() != 0;
}

} // namespace mrh

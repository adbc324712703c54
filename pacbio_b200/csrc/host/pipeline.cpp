#include "pipeline.hpp"
#include <chrono>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <map>
#include <stdexcept>
#include <sys/stat.h>
#include <unistd.h>
#include <cerrno>

namespace mrh {

std::vector<int> choose_devices() {
  std::vector<int> d;
  if(const char* e = getenv("MR_DEVICES")) {
    const char* p = e;
    while(*p) {
      char* end;
      const long v = strtol(p, &end, 10);
      if(end == p) break;
      d.push_back((int)v);
      p = *end ? end + 1 : end;
    }
  } else if(const char* g = getenv("MR_GPUS")) {
    for(int i = 0; i < atoi(g); ++i) d.push_back(i);
  }
  if(d.empty()) d.push_back(0);
  return d;
}

void build_indexes(device_set& ds, const std::vector<int>& devices, const super_reads& sr, const unitigs& u,
                   uint32_t psa_min, uint32_t mer) {
  ds.ctx.assign(devices.size(), nullptr);
  ds.idx.assign(devices.size(), nullptr);
  ds.owns_idx.assign(devices.size(), true);
  std::vector<std::string> errors(devices.size());
  std::vector<char> loaded(devices.size(), 0);
  // MR_INDEX_CACHE=<file>: reuse a saved index when it was built from these very inputs, else build
  // and save (the reference builds its suffix array again in every process)
  const char* cache = getenv("MR_INDEX_CACHE");
  const bool with_unitigs = !u.len.empty();
  const uint32_t* uid = with_unitigs ? sr.unitig_ids.data() : nullptr;
  const uint64_t* uoff = with_unitigs ? sr.unitig_off.data() : nullptr;
  const int32_t*  ulen = with_unitigs ? u.len.data() : nullptr;
  const uint64_t want = cache && *cache ? mr_inputs_checksum(sr.text2bit.data(), sr.n, sr.start.data(), sr.nseq(), uid, uoff, ulen,
                                                             (uint32_t)u.len.size(), psa_min, mer) : 0;
  std::vector<std::thread> th;
  for(size_t i = 0; i < devices.size(); ++i) {
    th.emplace_back([&, i]() {
      int rc = mr_context_create(devices[i], &ds.ctx[i]);
      if(rc != MR_OK) { errors[i] = std::string("mr_context_create: ") + mr_last_error(nullptr); return; }
      uint64_t on_disk = 0;
      if(cache && *cache && mr_index_peek_checksum(cache, &on_disk) == MR_OK && on_disk == want) {   // header first: no upload of a file for other inputs
        mr_index* got = nullptr;
        if(mr_index_load(ds.ctx[i], cache, &got) == MR_OK) {
          if(mr_index_checksum(got) == want) { ds.idx[i] = got; loaded[i] = 1; return; }
          mr_index_destroy(got);               // a file for other super-reads / options: ignore it
        }
      }
      rc = mr_index_create(ds.ctx[i], sr.text2bit.data(), sr.n, sr.start.data(), sr.nseq(), uid, uoff, ulen,
                           (uint32_t)u.len.size(), psa_min, mer, &ds.idx[i]);
      if(rc != MR_OK) errors[i] = std::string("mr_index_create: ") + mr_last_error(ds.ctx[i]);
    });
  }
  for(auto& t : th) t.join();
  for(const auto& e : errors) if(!e.empty()) throw std::runtime_error(e);
  if(cache && *cache) {
    if(loaded[0]) fprintf(stderr, "index: loaded from %s\n", cache);
    else {
      const std::string tmp = std::string(cache) + ".tmp";
      if(mr_index_save(ds.idx[0], tmp.c_str()) == MR_OK && rename(tmp.c_str(), cache) == 0) fprintf(stderr, "index: built and saved to %s\n", cache);
      else { remove(tmp.c_str()); fprintf(stderr, "index: built; could not save to %s\n", cache); }
    }
  }
}

unsigned streams_per_device() {
  if(const char* e = getenv("MR_STREAMS")) { const int v = atoi(e); return v < 1 ? 1u : (v > 8 ? 8u : (unsigned)v); }
  return 2;
}

bool stage_batches() {
  const char* e = getenv("MR_STAGE");
  return e && *e && *e != '0';
}

void add_streams(device_set& ds, unsigned per_device) {
  const size_t ndev = ds.ctx.size();
  for(unsigned s = 1; s < per_device; ++s) {
    for(size_t d = 0; d < ndev; ++d) {
      mr_context* c = nullptr;
      if(mr_context_create(mr_context_device(ds.ctx[d]), &c) != MR_OK) throw std::runtime_error(std::string("mr_context_create: ") + mr_last_error(nullptr));
      ds.ctx.push_back(c);
      ds.idx.push_back(ds.idx[d]);
      ds.owns_idx.push_back(false);
    }
  }
}

namespace {
struct part {
  std::unique_ptr<read_batch> batch;
  mr_result* result = nullptr;
  mr_text* text = nullptr;           // the part's records, when the device printed them
};
struct job {
  uint64_t seq = 0;                  // position in the input stream
  std::unique_ptr<read_batch> batch;
  std::vector<part> parts;           // aligned: one part, or several when the batch had to be split
};
}

namespace {
// Writes the text parts of one batch.  A regular file takes them through pwrite from one thread per part (each
// call copies its part into the page cache: a single writer tops out near 2 GB/s, a fraction of what the
// GPU produces); a pipe or terminal takes them in order through the stream.
struct record_writer {
  FILE* out;
  int   fd = -1;
  off_t at = 0;
  explicit record_writer(FILE* f) : out(f) {
    fflush(f);
    struct stat st;
    const int d = fileno(f);
    if(d >= 0 && fstat(d, &st) == 0 && S_ISREG(st.st_mode)) {
      const off_t cur = lseek(d, 0, SEEK_CUR);
      if(cur >= 0) { fd = d; at = cur; }
    }
  }
  struct span { const char* p; size_t n; };
  bool write(const std::vector<text_buf>& parts) {
    std::vector<span> sp;
    for(const auto& t : parts) sp.push_back(span{ t.data(), t.size() });
    return write(sp);
  }
  // one block of text, cut in pieces of at least 4 MB for the parallel writes
  bool write(const char* p, size_t n) {
    std::vector<span> sp;
    const size_t piece = std::max<size_t>(n / 8 + 1, 4u << 20);
    for(size_t o = 0; o < n; o += piece) sp.push_back(span{ p + o, std::min(piece, n - o) });
    return write(sp);
  }
  bool write(const std::vector<span>& parts) {
    if(fd < 0) {
      for(const auto& t : parts) if(t.n && fwrite(t.p, 1, t.n, out) != t.n) return false;
      return true;
    }
    std::vector<off_t> where(parts.size());
    for(size_t i = 0; i < parts.size(); ++i) { where[i] = at; at += (off_t)parts[i].n; }
    std::atomic<bool> ok(true);
    auto put = [&](size_t i) {
      const char* p = parts[i].p;
      size_t left = parts[i].n;
      off_t o = where[i];
      while(left) {
        const ssize_t w = pwrite(fd, p, left, o);
        if(w < 0) { if(errno == EINTR) continue; ok = false; return; }
        p += w; left -= (size_t)w; o += w;
      }
    };
    std::vector<std::thread> th;
    for(size_t i = 1; i < parts.size(); ++i) if(parts[i].n) th.emplace_back(put, i);
    if(!parts.empty() && parts[0].n) put(0);
    for(auto& t : th) t.join();
    return ok;
  }
  void finish() { if(fd >= 0) lseek(fd, at, SEEK_SET); }       // the stream's position follows what was written
};
}

uint64_t run_pipeline(device_set& ds, const std::vector<std::string>& read_paths, const mr_params& params,
                      const format_fn& format, FILE* out, unsigned host_threads, const records_fn& records) {
  // 32 Mbases per batch.  The library itself does better with 64 (bench.py's default: 9.8 against 9.1 Gbases/s on the
  // yeast shape, 0.84 against 0.66 on the human one -- fewer synchronisation points, twice the groups per launch of the
  // persistent chaining kernels), but the tools are bound by their reader (~2 Gbases/s), and page-locking the packed
  // arrays of the recycled batches (24 MB each at 64 Mbases; cudaHostRegister also holds up the kernel launches of
  // the aligner threads while it runs) only pays off over more batches than a short run has: create_mega_reads on
  // 0.6 Gbases of reads took 0.34 s with 32-Mbase batches and 1.5 s with 64.  MR_BATCH_BASES overrides.
  uint64_t batch_bases = 32ULL << 20;
  if(const char* e = getenv("MR_BATCH_BASES")) batch_bases = strtoull(e, nullptr, 0);
  const uint32_t batch_reads = 1u << 20;
  bounded_queue<job> to_align(2 * ds.ctx.size()), to_format(2 * ds.ctx.size());
  std::atomic<uint64_t> total_bases(0);
  std::string error;
  std::mutex error_mutex;
  std::atomic<bool> failed(false);       // what the worker threads test; the text stays under the mutex
  auto fail = [&](const std::string& msg) { std::lock_guard<std::mutex> l(error_mutex); if(error.empty()) error = msg; failed = true; };

  // Batches are recycled: a fresh one costs the reader 45 MB of first-touch page faults and zero fill (a third of its
  // time per batch); the formatter hands a batch back once its records are out.
  std::vector<std::unique_ptr<read_batch>> pool;
  std::mutex pool_mutex;
  auto now_us = []() { return (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  // Host -> device copies go through page-locked staging slots, two per context, locked ONCE (cudaHostRegister costs
  // 0.3-1.6 ms per MB depending on the host, and holds up the other threads' kernel launches while it runs): the
  // uploader thread copies a batch's packed arrays (0.375 bytes per base) into a free slot, the aligner's copy to the
  // device is then plain DMA.  Copying straight from the batch's pageable arrays made the driver stage the data itself,
  // next to a reader that faults pages in all the time: 20-40 ms per 13 MB batch.  MR_STAGE_SLOTS=0: pageable copies.
  struct pin_slot { uint64_t* codes = nullptr; uint64_t* nmask = nullptr; size_t ccap = 0, mcap = 0; };
  static const bool use_slots = !(getenv("MR_STAGE_SLOTS") && atoi(getenv("MR_STAGE_SLOTS")) == 0);
  std::vector<std::vector<pin_slot>> slots(ds.ctx.size(), std::vector<pin_slot>(2));
  std::vector<std::unique_ptr<bounded_queue<int>>> free_slots;
  for(size_t g = 0; g < ds.ctx.size(); ++g) {
    free_slots.emplace_back(new bounded_queue<int>(2));
    free_slots[g]->push(0); free_slots[g]->push(1);
  }
  auto slot_release = [&](size_t g, pin_slot& sl) {
    if(sl.codes) { mr_host_unpin(ds.ctx[g], sl.codes); free(sl.codes); sl.codes = nullptr; }
    if(sl.nmask) { mr_host_unpin(ds.ctx[g], sl.nmask); free(sl.nmask); sl.nmask = nullptr; }
    sl.ccap = sl.mcap = 0;
  };
  // copies the batch's packed arrays into the slot (grown and locked as needed); false: use the batch's own arrays
  auto slot_fill = [&](size_t g, pin_slot& sl, const read_batch& b) -> bool {
    const size_t cw = b.codes.size(), mw = b.nmask.size();
    if(cw > sl.ccap || mw > sl.mcap) {
      slot_release(g, sl);
      const size_t cc = cw + cw / 4 + 1024, mc = mw + mw / 4 + 1024;
      void *pc = nullptr, *pm = nullptr;
      if(posix_memalign(&pc, 4096, cc * 8) != 0 || posix_memalign(&pm, 4096, mc * 8) != 0) { free(pc); free(pm); return false; }
      if(mr_host_pin(ds.ctx[g], pc, cc * 8) != MR_OK) { free(pc); free(pm); return false; }
      if(mr_host_pin(ds.ctx[g], pm, mc * 8) != MR_OK) { mr_host_unpin(ds.ctx[g], pc); free(pc); free(pm); return false; }
      sl.codes = (uint64_t*)pc; sl.nmask = (uint64_t*)pm; sl.ccap = cc; sl.mcap = mc;
    }
    memcpy(sl.codes, b.codes.data(), cw * 8);
    memcpy(sl.nmask, b.nmask.data(), mw * 8);
    return true;
  };
  auto recycle = [&](std::unique_ptr<read_batch>& b) {
    if(!b) return;
    std::lock_guard<std::mutex> l(pool_mutex);
    if(pool.size() < 16) pool.push_back(std::move(b));
    else b.reset();
  };
  // MR_SHOW_TIMING: seconds every stage was busy (the stages overlap; the largest one bounds the phase)
  static const bool stage_timing = getenv("MR_SHOW_TIMING") != nullptr;
  std::atomic<uint64_t> busy_read_us(0), busy_upload_us(0), busy_align_us(0), busy_format_us(0), busy_write_us(0);

  std::thread reader([&]() {
    background_thread();
    try {
      read_stream rs(read_paths, host_threads);
      for(uint64_t seq = 0; ; ++seq) {
        job j;
        j.seq = seq;
        {
          std::lock_guard<std::mutex> l(pool_mutex);
          if(!pool.empty()) { j.batch = std::move(pool.back()); pool.pop_back(); }
        }
        if(!j.batch) j.batch.reset(new read_batch);
        j.batch->clear();
        const uint64_t t0 = now_us();
        const bool more = rs.next_batch(*j.batch, batch_bases, batch_reads, true);      // parsed and packed by the reader's workers
        busy_read_us += now_us() - t0;
        if(!more) break;
        total_bases += j.batch->bases.size();
        to_align.push(std::move(j));
      }
    } catch(std::exception& e) { fail(e.what()); }
    to_align.close();
  });

  // per context: an uploader thread stages the next batch (host -> device copy on the context's copy
  // stream, mr_stage_batch) while the aligner thread runs the kernels of the current one
  struct staged_job { job j; mr_staged* staged; int slot = -1; };
  std::vector<std::unique_ptr<bounded_queue<staged_job>>> staged;
  for(size_t g = 0; g < ds.ctx.size(); ++g) staged.emplace_back(new bounded_queue<staged_job>(1));
  std::vector<std::thread> aligners, uploaders;
  std::atomic<int> live((int)ds.ctx.size());
  for(size_t g = 0; g < ds.ctx.size(); ++g) {
    uploaders.emplace_back([&, g]() {
      job j;
      while(to_align.pop(j)) {
        staged_job sj;
        sj.staged = nullptr;
        const uint64_t t0 = now_us();
        if(!j.batch->packed()) j.batch->pack();  // 2 bits per base + non-ACGT mask: what crosses PCIe
        if(use_slots && !stage_batches()) {
          int k = -1;
          if(free_slots[g]->pop(k) && !slot_fill(g, slots[g][k], *j.batch)) { free_slots[g]->push(std::move(k)); k = -1; }
          sj.slot = k;
        }
        if(stage_batches() && !failed && mr_stage_batch_packed(ds.ctx[g], j.batch->codes.data(), j.batch->nmask.data(), j.batch->start.data(), j.batch->nreads(), &sj.staged) != MR_OK)
          sj.staged = nullptr;                  // the aligner retries through mr_align_batch and reports what is wrong
        busy_upload_us += now_us() - t0;
        sj.j = std::move(j);
        staged[g]->push(std::move(sj));
      }
      staged[g]->close();
    });
    aligners.emplace_back([&, g]() {
      staged_job sj;
      while(staged[g]->pop(sj)) {
        job j = std::move(sj.j);
        if(failed) { if(sj.staged) mr_staged_free(sj.staged); if(sj.slot >= 0) { int k = sj.slot; free_slots[g]->push(std::move(k)); } continue; }
        // A batch whose hits exceed a device limit (very repeat-rich reads) or the free memory is cut
        // in halves and retried; the halves are formatted in order, so the output does not change.
        std::deque<std::unique_ptr<read_batch>> work;
        work.push_back(std::move(j.batch));
        const uint64_t t0 = now_us();
        while(!work.empty() && !failed) {
          std::unique_ptr<read_batch> b = std::move(work.front());
          work.pop_front();
          part pt;
          int rc;
          if(sj.staged) { rc = mr_align_staged(ds.ctx[g], ds.idx[g], &params, sj.staged, &pt.result); sj.staged = nullptr; }
          else {
            if(!b->packed()) b->pack();         // a half of a batch that had to be split
            const bool from_slot = sj.slot >= 0;
            rc = mr_align_batch_packed(ds.ctx[g], ds.idx[g], &params, from_slot ? slots[g][sj.slot].codes : b->codes.data(),
                                       from_slot ? slots[g][sj.slot].nmask : b->nmask.data(), b->start.data(), b->nreads(), &pt.result);
            if(from_slot) { int k = sj.slot; sj.slot = -1; free_slots[g]->push(std::move(k)); }    // (a batch that is split is retried from its own arrays)
          }
          if(rc == MR_OK) {
            if(records) {                       // printed on the device while the rows are still there
              try { pt.text = records(ds.ctx[g], pt.result, *b); } catch(std::exception& e) { fail(e.what()); }
            }
            pt.batch = std::move(b);
            j.parts.push_back(std::move(pt));
            continue;
          }
          if((rc == MR_ELIMIT || rc == MR_ENOMEM) && b->nreads() > 1) {
            const uint32_t half = b->nreads() / 2;
            std::unique_ptr<read_batch> lo(new read_batch), hi(new read_batch);
            lo->bases.assign(b->bases, 0, b->start[half]);
            lo->start.assign(b->start.begin(), b->start.begin() + half + 1);
            lo->name.assign(b->name.begin(), b->name.begin() + half);
            hi->bases.assign(b->bases, b->start[half], std::string::npos);
            for(uint32_t r = half; r <= b->nreads(); ++r) hi->start.push_back(b->start[r] - b->start[half]);
            hi->name.assign(b->name.begin() + half, b->name.end());
            work.push_front(std::move(hi));
            work.push_front(std::move(lo));
            continue;
          }
          fail(std::string("mr_align_batch: ") + mr_last_error(ds.ctx[g]));
        }
        busy_align_us += now_us() - t0;
        to_format.push(std::move(j));
      }
      if(--live == 0) to_format.close();
    });
  }

  std::thread formatter([&]() {
    background_thread();                       // (and so are the threads it starts: a new thread inherits the nice value)
    job j;
    std::vector<text_buf> parts;
    record_writer writer(out);
    std::map<uint64_t, job> waiting;           // aligned out of turn (several aligner threads)
    uint64_t next_seq = 0;
    while(to_format.pop(j)) {
      waiting.emplace(j.seq, std::move(j));
      for(auto it = waiting.find(next_seq); it != waiting.end(); it = waiting.find(++next_seq)) {
        for(auto& pt : it->second.parts) {
          const uint64_t t0 = now_us();
          bool ok = true;
          if(pt.text) {
            const char* p = nullptr;
            uint64_t n = 0;
            mr_text_get(pt.text, &p, &n);
            ok = writer.write(p, n);
            mr_text_free(pt.text);
            busy_write_us += now_us() - t0;
          } else if(!failed) {
            mr_result_view v;
            mr_result_get(pt.result, &v);
            for(auto& p : parts) p.clear();
            try { format(pt.result, v, *pt.batch, parts); } catch(std::exception& e) { fail(e.what()); }
            const uint64_t t1 = now_us();
            ok = failed || writer.write(parts);
            busy_format_us += t1 - t0; busy_write_us += now_us() - t1;
          }
          if(!ok) fail("write error on output file");
          mr_result_free(pt.result);
          recycle(pt.batch);
        }
        waiting.erase(it);
      }
    }
    for(auto& w : waiting) for(auto& pt : w.second.parts) { mr_text_free(pt.text); mr_result_free(pt.result); }   // only after an error
    writer.finish();
  });

  reader.join();
  for(auto& t : uploaders) t.join();
  for(auto& t : aligners) t.join();
  formatter.join();
  fflush(out);
  for(size_t g = 0; g < ds.ctx.size(); ++g) for(auto& sl : slots[g]) slot_release(g, sl);
  if(stage_timing)
    fprintf(stderr, "stage busy seconds (overlapping): read+pack %.3f, upload %.3f (%zu threads), align %.3f (%zu threads), format %.3f, write %.3f\n",
            1e-6 * busy_read_us, 1e-6 * busy_upload_us, ds.ctx.size(), 1e-6 * busy_align_us, ds.ctx.size(), 1e-6 * busy_format_us, 1e-6 * busy_write_us);
  if(!error.empty()) throw std::runtime_error(error);
  return total_bases;
}

namespace {
// names back to back and their offsets, as the C ABI takes them
void join_names(const std::vector<std::string>& names, std::string& all, std::vector<uint64_t>& off) {
  off.assign(1, 0);
  off.reserve(names.size() + 1);
  for(const auto& n : names) { all += n; off.push_back(all.size()); }
}
}

mr_text* device_records(mr_context* ctx, const mr_result* r, const mr_records_params& p, const mr_unitigs* u,
                        const std::vector<std::string>& names) {
  std::string all;
  std::vector<uint64_t> off;
  join_names(names, all, off);
  mr_text* t = nullptr;
  if(mr_records(ctx, r, &p, u, all.data(), off.data(), &t) != MR_OK) throw std::runtime_error(mr_last_error(ctx));
  return t;
}

mr_text* device_coords(mr_context* ctx, const mr_result* r, const mr_coords_params& p, const mr_sr_names* s,
                       const std::vector<std::string>& names) {
  std::string all;
  std::vector<uint64_t> off;
  join_names(names, all, off);
  mr_text* t = nullptr;
  if(mr_coords_records(ctx, r, &p, s, all.data(), off.data(), &t) != MR_OK) throw std::runtime_error(mr_last_error(ctx));
  return t;
}

void device_sr_names::upload(const device_set& ds, const super_reads& SR) {
  std::string all;
  std::vector<uint64_t> off;
  join_names(SR.name, all, off);
  for(mr_context* c : ds.ctx) {
    const int d = mr_context_device(c);
    if(std::find(device.begin(), device.end(), d) != device.end()) continue;
    mr_sr_names* x = nullptr;
    if(mr_sr_names_create(c, all.data(), off.data(), SR.unitig_ids.empty() ? nullptr : SR.unitig_ids.data(), SR.unitig_off.data(),
                          SR.nseq(), &x) != MR_OK)
      throw std::runtime_error(std::string("mr_sr_names_create: ") + mr_last_error(c));
    device.push_back(d);
    s.push_back(x);
  }
}

const mr_sr_names* device_sr_names::of(mr_context* ctx) const {
  const int d = mr_context_device(ctx);
  for(size_t i = 0; i < device.size(); ++i) if(device[i] == d) return s[i];
  return nullptr;
}

void device_unitigs::upload(const device_set& ds, const unitigs& U) {
  if(!U.has_sequences()) return;
  for(mr_context* c : ds.ctx) {
    const int d = mr_context_device(c);
    if(std::find(device.begin(), device.end(), d) != device.end()) continue;
    mr_unitigs* x = nullptr;
    if(mr_unitigs_create(c, U.fwd.data(), U.off.data(), (uint32_t)U.len.size(), &x) != MR_OK)
      throw std::runtime_error(std::string("mr_unitigs_create: ") + mr_last_error(c));
    device.push_back(d);
    u.push_back(x);
  }
}

const mr_unitigs* device_unitigs::of(mr_context* ctx) const {
  const int d = mr_context_device(ctx);
  for(size_t i = 0; i < device.size(); ++i) if(device[i] == d) return u[i];
  return nullptr;
}

mr_records_params records_params(const graph_options& g) {
  mr_records_params p;
  p.unitigs_k = g.k_len; p.overlap_play = g.overlap_play; p.density = g.density; p.min_length = g.min_length;
  p.tiling = g.tiling; p.trim = g.trim;
  return p;
}

} // namespace mrh

// Batch pipeline shared by the two tools: a reader thread cuts the long-read stream into batches,
// one aligner thread per GPU context pushes them through the C ABI, a formatter stage turns each
// result into text (fanned out over -t host threads) and writes the records in input order.  Reads are
// partitioned across GPUs batch by batch with the index replicated per GPU; there is no
// collective on the path, only this host-side gather (SURVEY.md 8e).
#pragma once
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>

#include "host_common.hpp"

namespace mrh {

template<typename T>
class bounded_queue {
  std::deque<T> q_;
  std::mutex m_;
  std::condition_variable cv_push_, cv_pop_;
  size_t cap_;
  bool closed_ = false;
public:
  explicit bounded_queue(size_t cap) : cap_(cap) { }
  void push(T&& x) {
    std::unique_lock<std::mutex> l(m_);
    cv_push_.wait(l, [&] { return q_.size() < cap_; });
    q_.push_back(std::move(x));
    cv_pop_.notify_one();
  }
  bool pop(T& x) {
    std::unique_lock<std::mutex> l(m_);
    cv_pop_.wait(l, [&] { return !q_.empty() || closed_; });
    if(q_.empty()) return false;
    x = std::move(q_.front());
    q_.pop_front();
    cv_push_.notify_one();
    return true;
  }
  void close() { std::lock_guard<std::mutex> l(m_); closed_ = true; cv_pop_.notify_all(); }
};

// one entry per aligner thread: a context (stream + scratch) and the index it reads.  Several
// contexts of one device share that device's index (owns_idx false for all but the first).
struct device_set {
  std::vector<mr_context*> ctx;
  std::vector<mr_index*>   idx;
  std::vector<bool>        owns_idx;
  ~device_set() {
    for(size_t i = 0; i < idx.size(); ++i) if(i >= owns_idx.size() || owns_idx[i]) mr_index_destroy(idx[i]);
    for(auto c : ctx) mr_context_destroy(c);
  }
};

// devices from MR_DEVICES ("0,1,2"), MR_GPUS (count) or just device 0
std::vector<int> choose_devices();

// creates one context + index per device (index build runs concurrently on all of them)
void build_indexes(device_set& ds, const std::vector<int>& devices, const super_reads& sr, const unitigs& u,
                   uint32_t psa_min, uint32_t mer);

// batches in flight per device: MR_STREAMS (default 2).  The kernels of one batch are a mix of
// bandwidth-bound (seed lookups, sort) and latency-bound (chaining, coords) work with host round
// trips in between; a second batch on its own stream fills those gaps (measured on B200, configs[1]:
// device 85.7 -> 77.5 ms per step, end to end 90.9 -> 81.0).  In round 1 the end-to-end rate DROPPED with a
// second stream because its aligner thread took a core from the threads that tile and print the records;
// that stage costs half as much now (exact integer formatter, sequence arena).
unsigned streams_per_device();
// adds per_device - 1 more contexts for every device of ds, sharing the device's index
void add_streams(device_set& ds, unsigned per_device);

// format(result, view, batch, parts): the batch's text in parts[], written by the pipeline when it returns (host
// formatting, on the one formatter thread)
typedef std::function<void(const mr_result*, const mr_result_view&, const read_batch&, std::vector<text_buf>&)> format_fn;
// records(context, result, batch): the batch's text produced on the device (mr_records, mr_coords_records), called by the aligner
// thread of `context` right after the batch is aligned, while its rows are still on the device.  When given, it
// replaces `format` and the formatter thread only writes the text; it throws std::runtime_error on failure.
typedef std::function<mr_text*(mr_context*, const mr_result*, const read_batch&)> records_fn;

// runs the whole stream; returns the number of read bases processed
// host_threads: workers of the reader (parsing, packing); 0 = as many as the box has, up to 16
uint64_t run_pipeline(device_set& ds, const std::vector<std::string>& read_paths, const mr_params& params,
                      const format_fn& format, FILE* out, unsigned host_threads = 0, const records_fn& records = records_fn());

// mr_records over a batch of a tool: the reads' names as the C ABI takes them, errors as exceptions
mr_text* device_records(mr_context* ctx, const mr_result* r, const mr_records_params& p, const mr_unitigs* u,
                        const std::vector<std::string>& names);
// the -u sequences on every device of ds (one upload per device, shared by its contexts); empty without -u
struct device_unitigs {
  std::vector<int> device;
  std::vector<mr_unitigs*> u;
  ~device_unitigs() { for(auto x : u) mr_unitigs_destroy(x); }
  void upload(const device_set& ds, const unitigs& U);
  const mr_unitigs* of(mr_context* ctx) const;
};
mr_records_params records_params(const graph_options& g);

// mr_coords_records over a batch of a tool: the reads' names as the C ABI takes them, errors as exceptions
mr_text* device_coords(mr_context* ctx, const mr_result* r, const mr_coords_params& p, const mr_sr_names* s,
                       const std::vector<std::string>& names);
// the super-reads' names and paths on every device of ds (one upload per device, shared by its contexts)
struct device_sr_names {
  std::vector<int> device;
  std::vector<mr_sr_names*> s;
  ~device_sr_names() { for(auto x : s) mr_sr_names_destroy(x); }
  void upload(const device_set& ds, const super_reads& SR);
  const mr_sr_names* of(mr_context* ctx) const;
};

} // namespace mrh

// same_multi.cu — one receiver batch sharded over several CUDA devices inside ONE process: one host thread, one engine
// and one pair of CUDA streams per device (BASELINE.json north_star: "streams shard naturally across the 8 GPUs of one
// box, with one host thread and CUDA stream per device"; SURVEY.md §8e).
//
// Streams are independent (SameReceiver owns all of its state, receiver.rs:71-90), so there is no collective and no
// device-to-device traffic: shard i owns the contiguous stream range [first_i, first_i + count_i), every call fans out
// to the shards' worker threads, and drain concatenates the per-device event lists re-tagged with global stream ids
// (the "host-side gather of decoded messages").  Built on the public single-device C ABI, plus the engine's internal
// stream-state helpers (same_engine.cu) so that an import can validate on every shard before any shard changes.
#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "same_internal.h"

namespace {

struct Shard {
  int device = 0;
  uint32_t first = 0, count = 0;
  same_engine* eng = nullptr;
  // worker thread + one-slot mailbox
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  bool has_job = false, done = true, quit = false;
  int rc = 0;
  // scratch reused across submits
  std::vector<uint64_t> off;
  std::vector<uint32_t> map;   // interleaved submit: this shard's stream of each channel
  size_t pend_ev = 0, pend_pay = 0;
  // stream-state export / import: this shard's share of a call
  std::vector<uint32_t> st_ids, st_pos;
  std::vector<uint8_t> st_buf;
  uint32_t st_flags = 0;
  std::string err;   // text of a failed create (the library's last-error string is per thread)
};

void worker_main(Shard* s) {
  std::unique_lock<std::mutex> lk(s->mu);
  while (true) {
    s->cv.wait(lk, [&] { return s->has_job || s->quit; });
    if (s->quit) return;
    std::function<int()> job = std::move(s->job);
    s->has_job = false;
    lk.unlock();
    const int rc = job();
    lk.lock();
    s->rc = rc;
    s->done = true;
    s->cv.notify_all();
  }
}

}  // namespace

struct same_multi {
  std::vector<Shard*> shards;
  uint32_t n_streams = 0;
  std::string last_error;
};

namespace {

thread_local std::string g_multi_error;

int mfail(same_multi* m, int code, const std::string& msg) {
  if (m) m->last_error = msg;
  g_multi_error = msg;
  return code;
}

// Run fn(shard) on every shard's own thread, wait for all, return the first non-zero status (with that engine's text).
int run_all(same_multi* m, const std::function<int(Shard&)>& fn) {
  for (Shard* s : m->shards) {
    std::lock_guard<std::mutex> lk(s->mu);
    s->job = [s, &fn]() { return fn(*s); };
    s->has_job = true; s->done = false;
    s->cv.notify_all();
  }
  int rc = SAME_OK;
  for (Shard* s : m->shards) {
    std::unique_lock<std::mutex> lk(s->mu);
    s->cv.wait(lk, [&] { return s->done; });
    if (s->rc != SAME_OK && rc == SAME_OK) {
      rc = s->rc;
      m->last_error = "device " + std::to_string(s->device) + " (streams " + std::to_string(s->first) + ".." +
                      std::to_string(s->first + s->count) + "): " + (s->eng ? same_engine_last_error(s->eng) : s->err.c_str());
    }
  }
  return rc;
}

}  // namespace

extern "C" {

const char* same_multi_last_error(const same_multi* m) { return m ? m->last_error.c_str() : g_multi_error.c_str(); }

int same_multi_create(const same_config* cfg, const int* devices, uint32_t n_devices, uint32_t n_streams,
                      same_multi** out) {
  if (!cfg || !devices || !out || n_devices == 0) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (n_streams < n_devices) return mfail(nullptr, SAME_ERR_INVALID_ARG, "fewer streams than devices");
  same_multi* m = new same_multi();
  m->n_streams = n_streams;
  for (uint32_t i = 0; i < n_devices; ++i) {
    Shard* s = new Shard();
    s->device = devices[i];
    s->first = (uint32_t)((uint64_t)n_streams * i / n_devices);
    s->count = (uint32_t)((uint64_t)n_streams * (i + 1) / n_devices) - s->first;
    m->shards.push_back(s);
    s->th = std::thread(worker_main, s);
  }
  // engines are created on their own threads (context creation per device runs in parallel)
  const int rc = run_all(m, [cfg](Shard& s) {
    const int r = same_engine_create(cfg, s.device, s.count, &s.eng);
    if (r != SAME_OK) s.err = same_last_error();
    return r;
  });
  if (rc != SAME_OK) {
    g_multi_error = m->last_error;
    same_multi_destroy(m);
    return rc;
  }
  *out = m;
  return SAME_OK;
}

void same_multi_destroy(same_multi* m) {
  if (!m) return;
  for (Shard* s : m->shards) {
    if (s->eng) {
      std::lock_guard<std::mutex> lk(s->mu);
      same_engine* e = s->eng;
      s->job = [e]() { same_engine_destroy(e); return 0; };
      s->has_job = true; s->done = false; s->eng = nullptr;
      s->cv.notify_all();
    }
  }
  for (Shard* s : m->shards) {
    {
      std::unique_lock<std::mutex> lk(s->mu);
      s->cv.wait(lk, [&] { return s->done; });
      s->quit = true;
      s->cv.notify_all();
    }
    if (s->th.joinable()) s->th.join();
    delete s;
  }
  delete m;
}

uint32_t same_multi_num_shards(const same_multi* m) { return m ? (uint32_t)m->shards.size() : 0u; }
uint32_t same_multi_num_streams(const same_multi* m) { return m ? m->n_streams : 0u; }

int same_multi_shard_info(const same_multi* m, uint32_t shard, int* device, uint32_t* first_stream, uint32_t* n_streams) {
  if (!m || shard >= m->shards.size()) return SAME_ERR_INVALID_ARG;
  if (device) *device = m->shards[shard]->device;
  if (first_stream) *first_stream = m->shards[shard]->first;
  if (n_streams) *n_streams = m->shards[shard]->count;
  return SAME_OK;
}

same_engine* same_multi_engine(same_multi* m, uint32_t shard) {
  return (m && shard < m->shards.size()) ? m->shards[shard]->eng : nullptr;
}

// Each device copies only the span of the host buffer its own streams touch.
static int multi_submit_flat(same_multi* m, const void* samples, int fmt, uint64_t total, const uint64_t* offsets,
                             const uint32_t* lengths) {
  if (!m || !offsets || !lengths || (!samples && total)) return mfail(m, SAME_ERR_INVALID_ARG, "null argument");
  for (uint32_t i = 0; i < m->n_streams; ++i)
    if (lengths[i] && offsets[i] + lengths[i] > total) return mfail(m, SAME_ERR_INVALID_ARG, "offset+length exceeds total_samples");
  return run_all(m, [=](Shard& s) {
    uint64_t lo = UINT64_MAX, hi = 0;
    for (uint32_t i = s.first; i < s.first + s.count; ++i)
      if (lengths[i]) { lo = std::min(lo, offsets[i]); hi = std::max(hi, offsets[i] + lengths[i]); }
    if (hi == 0) lo = 0;
    s.off.resize(s.count);
    for (uint32_t i = 0; i < s.count; ++i) s.off[i] = lengths[s.first + i] ? offsets[s.first + i] - lo : 0;
    if (fmt == 1)
      return same_engine_submit_f32(s.eng, static_cast<const float*>(samples) + lo, hi - lo, s.off.data(), lengths + s.first);
    return same_engine_submit_s16(s.eng, static_cast<const int16_t*>(samples) + lo, hi - lo, s.off.data(), lengths + s.first);
  });
}

int same_multi_submit_s16(same_multi* m, const int16_t* samples, uint64_t total_samples, const uint64_t* offsets,
                          const uint32_t* lengths) {
  return multi_submit_flat(m, samples, 0, total_samples, offsets, lengths);
}

int same_multi_submit_f32(same_multi* m, const float* samples, uint64_t total_samples, const uint64_t* offsets,
                          const uint32_t* lengths) {
  return multi_submit_flat(m, samples, 1, total_samples, offsets, lengths);
}

int same_multi_submit_s16_2d(same_multi* m, const int16_t* samples, uint64_t row_stride, uint64_t col_start,
                             uint32_t n_cols) {
  if (!m || !samples) return mfail(m, SAME_ERR_INVALID_ARG, "null argument");
  return run_all(m, [=](Shard& s) {
    return same_engine_submit_s16_2d(s.eng, samples + (uint64_t)s.first * row_stride, row_stride, col_start, n_cols);
  });
}

// Every shard sees the whole frames with a map of its own streams only, so its engine copies and converts just the
// column range of its own channels.
int same_multi_submit_interleaved(same_multi* m, const void* frames, uint32_t format, uint32_t n_channels,
                                  uint64_t n_frames, const uint32_t* channel_stream) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  std::string why;
  if (same_check_interleaved(frames, format, n_channels, n_frames, channel_stream, m->n_streams, &why))
    return mfail(m, SAME_ERR_INVALID_ARG, why);
  return run_all(m, [=](Shard& s) {
    s.map.resize(n_channels);
    for (uint32_t c = 0; c < n_channels; ++c) {
      const uint32_t g = channel_stream ? channel_stream[c] : c;
      s.map[c] = g != SAME_CHANNEL_SKIP && g >= s.first && g - s.first < s.count ? g - s.first : SAME_CHANNEL_SKIP;
    }
    return same_engine_submit_interleaved(s.eng, frames, format, n_channels, n_frames, s.map.data());
  });
}

int same_multi_submit_zeros(same_multi* m, const uint32_t* lengths) {
  if (!m || !lengths) return mfail(m, SAME_ERR_INVALID_ARG, "null argument");
  return run_all(m, [=](Shard& s) { return same_engine_submit_zeros(s.eng, lengths + s.first); });
}

int same_multi_sync(same_multi* m) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  return run_all(m, [](Shard& s) { return same_engine_sync(s.eng); });
}

int same_multi_reset(same_multi* m) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  return run_all(m, [](Shard& s) { return same_engine_reset(s.eng, nullptr, 0); });
}

int same_multi_input_sample_counters(same_multi* m, uint64_t* out) {
  if (!m || !out) return mfail(m, SAME_ERR_INVALID_ARG, "null argument");
  return run_all(m, [=](Shard& s) { return same_engine_input_sample_counters(s.eng, out + s.first); });
}

int same_multi_pending(same_multi* m, size_t* n_events, size_t* n_payload_bytes) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  const int rc = run_all(m, [](Shard& s) { return same_engine_pending(s.eng, &s.pend_ev, &s.pend_pay); });
  size_t ne = 0, np = 0;
  for (Shard* s : m->shards) { ne += s->pend_ev; np += s->pend_pay; }
  if (n_events) *n_events = ne;
  if (n_payload_bytes) *n_payload_bytes = np;
  return rc;
}

// All pending events of all devices, sorted by (global stream, order of occurrence): shards are contiguous and each
// engine hands its events out sorted, so the concatenation in shard order is the global order.
int same_multi_drain_events(same_multi* m, same_event* events, size_t events_cap, size_t* n_events, uint8_t* payload,
                            size_t payload_cap, size_t* n_payload) {
  size_t ne = 0, np = 0;
  int rc = same_multi_pending(m, &ne, &np);
  if (rc != SAME_OK) return rc;
  if (n_events) *n_events = ne;
  if (n_payload) *n_payload = np;
  if (ne > events_cap || np > payload_cap || (ne && !events) || (np && !payload))
    return mfail(m, SAME_ERR_INVALID_ARG, "drain buffers too small");
  std::vector<size_t> ev_base(m->shards.size()), pay_base(m->shards.size());
  size_t e0 = 0, p0 = 0;
  for (size_t i = 0; i < m->shards.size(); ++i) {
    ev_base[i] = e0; pay_base[i] = p0;
    e0 += m->shards[i]->pend_ev; p0 += m->shards[i]->pend_pay;
  }
  std::vector<Shard*>& sh = m->shards;
  return run_all(m, [&](Shard& s) {
    size_t i = 0;
    while (sh[i] != &s) ++i;
    size_t a = 0, b = 0;
    same_event* dst = events ? events + ev_base[i] : nullptr;
    const int r = same_engine_drain_events(s.eng, dst, s.pend_ev, &a, payload ? payload + pay_base[i] : nullptr, s.pend_pay, &b);
    if (r != SAME_OK) return r;
    for (size_t k = 0; k < a; ++k) { dst[k].stream += s.first; dst[k].data_offset += (uint32_t)pay_base[i]; }
    return (int)SAME_OK;
  });
}

// ---- portable stream state with global ids ----
size_t same_multi_state_bytes(const same_multi* m, uint32_t n) {
  return m ? same_state_engine_header_bytes(m->shards[0]->eng) + (size_t)n * same_state_engine_record_bytes(m->shards[0]->eng) : 0;
}

// ids -> each shard's local ids and positions in `ids`; false on an id out of range (or a duplicate, if unique)
static bool split_ids(same_multi* m, const uint32_t* ids, uint32_t n, bool unique) {
  for (Shard* s : m->shards) { s->st_ids.clear(); s->st_pos.clear(); }
  std::vector<char> seen(unique ? m->n_streams : 0, 0);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t g = ids ? ids[i] : i;
    if (g >= m->n_streams) { mfail(m, SAME_ERR_INVALID_ARG, "stream id " + std::to_string(g) + " out of range"); return false; }
    if (unique) {
      if (seen[g]) { mfail(m, SAME_ERR_INVALID_ARG, "duplicate target stream id " + std::to_string(g)); return false; }
      seen[g] = 1;
    }
    size_t k = 0;
    while (g >= m->shards[k]->first + m->shards[k]->count) ++k;
    m->shards[k]->st_ids.push_back(g - m->shards[k]->first);
    m->shards[k]->st_pos.push_back(i);
  }
  return true;
}

int same_multi_export_streams(same_multi* m, const uint32_t* ids, uint32_t n, void* buf, size_t cap, size_t* written) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  if (!ids) n = m->n_streams;
  if (!split_ids(m, ids, n, false)) return SAME_ERR_INVALID_ARG;
  const size_t need = same_multi_state_bytes(m, n);
  if (written) *written = need;
  if (!buf || cap < need) return mfail(m, SAME_ERR_INVALID_ARG, "export buffer too small: " + std::to_string(need) + " bytes needed");
  const size_t hdr = same_state_engine_header_bytes(m->shards[0]->eng), rec = same_state_engine_record_bytes(m->shards[0]->eng);
  same_state_write_header(m->shards[0]->eng, n, buf);
  uint8_t* out = static_cast<uint8_t*>(buf) + hdr;
  return run_all(m, [=](Shard& s) {
    const uint32_t k = (uint32_t)s.st_ids.size();
    if (k == 0) return (int)SAME_OK;
    // records of a run of consecutive positions go straight to their place in the caller's buffer
    const bool in_place = s.st_pos.back() - s.st_pos.front() + 1u == k;
    uint8_t* dst = out + (size_t)s.st_pos.front() * rec;
    if (!in_place) { s.st_buf.resize((size_t)k * rec); dst = s.st_buf.data(); }
    const int r = same_state_export_records(s.eng, s.st_ids.data(), k, s.first, dst);
    if (r != SAME_OK || in_place) return r;
    for (uint32_t j = 0; j < k; ++j) memcpy(out + (size_t)s.st_pos[j] * rec, s.st_buf.data() + (size_t)j * rec, rec);
    return (int)SAME_OK;
  });
}

int same_multi_import_streams(same_multi* m, const uint32_t* ids, uint32_t n, const void* buf, size_t len) {
  if (!m) return mfail(nullptr, SAME_ERR_INVALID_ARG, "null handle");
  uint32_t n_records = 0;
  same_engine* e0 = m->shards[0]->eng;
  int rc = same_state_check_header(e0, buf, len, &n_records);   // every shard has the same configuration
  if (rc != SAME_OK) return mfail(m, rc, same_engine_last_error(e0));
  if (!ids && n != m->n_streams) return mfail(m, SAME_ERR_INVALID_ARG, "ids == NULL imports into every stream: n must equal the number of streams");
  if (n != n_records) return mfail(m, SAME_ERR_INVALID_ARG, "n = " + std::to_string(n) + " but the buffer holds " + std::to_string(n_records) + " records");
  if (!split_ids(m, ids, n, true)) return SAME_ERR_INVALID_ARG;
  const size_t hdr = same_state_engine_header_bytes(e0), rec = same_state_engine_record_bytes(e0);
  const uint8_t* in = static_cast<const uint8_t*>(buf) + hdr;
  // every shard stages and validates its records; only if all of them passed does any shard write its streams
  rc = run_all(m, [=](Shard& s) {
    const uint32_t k = (uint32_t)s.st_ids.size();
    if (k == 0) return (int)SAME_OK;
    const uint8_t* src = in + (size_t)s.st_pos.front() * rec;
    if (s.st_pos.back() - s.st_pos.front() + 1u != k) {
      s.st_buf.resize((size_t)k * rec);
      for (uint32_t j = 0; j < k; ++j) memcpy(s.st_buf.data() + (size_t)j * rec, in + (size_t)s.st_pos[j] * rec, rec);
      src = s.st_buf.data();
    }
    return same_state_import_stage(s.eng, k, src, &s.st_flags);
  });
  if (rc != SAME_OK) return rc;
  return run_all(m, [](Shard& s) {
    const uint32_t k = (uint32_t)s.st_ids.size();
    return k ? same_state_import_commit(s.eng, s.st_ids.data(), k, s.st_flags) : (int)SAME_OK;
  });
}

}  // extern "C"

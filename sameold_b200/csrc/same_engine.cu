// same_engine.cu — host side of the C ABI declared in include/same_engine.h.
//
// Responsibilities: configuration clamping (builder.rs setters), derivation of the receiver constants exactly as
// SameReceiver::from does (receiver.rs:502-560; libm cosf/sinf/expf/sinhf on the host, bits uploaded to the device),
// device memory for the resident per-stream state, double-buffered host->device sample copies overlapped with the
// receiver kernel, and the event arena -> host hand-off.  There is no CPU decode path in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "same_internal.h"

namespace {

thread_local std::string g_last_error;

// Rust f32::clamp / min / max semantics for the builder setters
inline float rclampf(float x, float lo, float hi) { if (x < lo) x = lo; if (x > hi) x = hi; return x; }

constexpr float kMarkHz = 2083.3f;    // waveform.rs:6
constexpr float kSpaceHz = 1562.5f;   // waveform.rs:9
constexpr float kBaudHz = 520.83f;    // waveform.rs:12
constexpr float kPi = 3.14159265358979323846f;  // std::f32::consts::PI

// waveform.rs:54-64: h[i] = 2 * conj(exp(j*2*pi*f*(N-1-i))) / N, all in f32
void cisoid_taps(uint32_t n, float freq_fs, float* re, float* im) {
  for (uint32_t i = 0; i < n; ++i) {
    float th = 2.0f * kPi * freq_fs * (float)(n - 1 - i);
    float r = expf(0.0f);
    float c = r * cosf(th), s = r * sinf(th);
    re[i] = (2.0f * c) / (float)n;
    im[i] = (2.0f * (-s)) / (float)n;
  }
}

// symsync.rs:329-337
void loop_alphabeta(float bw, float& alpha, float& beta) {
  float w = 2.0f * kPi * bw;
  float k0 = 2.0f, k1 = expf(-w), sh = sinhf(w);
  alpha = k0 * k1 * sh;
  beta = k0 * (1.0f - k1 * (sh + 1.0f));
}

// The input rates whose matched filter has 1..max_taps taps, in the engine's own f32 arithmetic (same_ntaps)
void rate_range(size_t max_taps, uint32_t* lo, uint32_t* hi) {
  uint32_t r = 1;
  while (same_ntaps(r) < 1) ++r;
  *lo = r;
  r = (uint32_t)((double)(max_taps + 1) * kBaudHz) + 2u;
  while (same_ntaps(r) > max_taps) --r;
  while (same_ntaps(r + 1) <= max_taps) ++r;
  *hi = r;
}

// ---- owned CUDA resources: released when their owner goes, on the device that is current then ----

// An array of T from Alloc, released with Free.  grow() allocates before it releases: a failed allocation leaves the
// old array in place and clears the runtime's last error, so that the next launcher does not report it as its own.
template <class T, cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
class Buf {
 public:
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  ~Buf() { if (p_) Free(p_); }
  operator T*() const { return p_; }
  size_t size() const { return n_; }   // elements
  // room for at least n elements (when it has to grow: n + slack); the contents are not kept
  cudaError_t grow(size_t n, size_t slack = 0) {
    if (n <= n_) return cudaSuccess;
    void* q = nullptr;
    const cudaError_t err = Alloc(&q, (n + slack) * sizeof(T));
    if (err != cudaSuccess) { cudaGetLastError(); return err; }
    if (p_) Free(p_);
    p_ = static_cast<T*>(q); n_ = n + slack;
    return cudaSuccess;
  }
  void swap(Buf& o) { std::swap(p_, o.p_); std::swap(n_, o.n_); }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};
template <class T> using DevBuf = Buf<T, cudaMalloc, cudaFree>;
template <class T> using PinnedBuf = Buf<T, cudaMallocHost, cudaFreeHost>;

class Event {
 public:
  Event() = default;
  Event(const Event&) = delete;
  Event& operator=(const Event&) = delete;
  ~Event() { if (ev_) cudaEventDestroy(ev_); }
  cudaError_t create(unsigned flags = cudaEventDefault) { return cudaEventCreateWithFlags(&ev_, flags); }
  operator cudaEvent_t() const { return ev_; }

 private:
  cudaEvent_t ev_ = nullptr;
};

class Stream {
 public:
  Stream() = default;
  Stream(const Stream&) = delete;
  Stream& operator=(const Stream&) = delete;
  ~Stream() { if (st_) cudaStreamDestroy(st_); }
  cudaError_t create() { return cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking); }
  operator cudaStream_t() const { return st_; }

 private:
  cudaStream_t st_ = nullptr;
};

struct InputBuf {
  DevBuf<uint8_t> d;                     // device samples (s16 or f32)
  DevBuf<unsigned long long> d_off;
  DevBuf<uint32_t> d_len;
  Event copied, consumed;
  bool used = false;
};

}  // namespace

struct same_engine {
  Stream compute, copy;   // declared first, so destroyed last
  same_config cfg;
  int device = 0;
  uint32_t n_streams = 0;
  SameParams p;           // its pointers into the buffers below are set by bind()
  SameTapsWide taps_wide;   // every tap: the wide kernel's, the state header's and same_engine_get_derived's
  SameTaps taps;            // the first SAME_GENERIC_TAPS of them for the generic kernel
  SameTaps2 taps2;
  Kernel kernel_override = POLICY;   // option "kernel"
  uint32_t lanes_per_warp = 32;   // streams per warp in the fast kernel (lane-sparse warps for small batches)
  int sm_count = 148;
  // split pipeline (kernel 5): front-end output, allocated on first use
  SameTiles tiles{nullptr, nullptr, 0u, 32u, 1u};
  DevBuf<float> tiles_d;
  DevBuf<uint32_t> tiles_dc_next;
  // long-stream path (same_long.cu): one stream, long chunks
  int long_stream = 1;            // option "long_stream"
  DevBuf<float> ls_d, ls_y, ls_g, ls_soft, ls_gin;
  DevBuf<uint32_t> ls_ctrl;       // {verified end, position reached, reason, span length}
  DevBuf<unsigned long long> ls_off;   // offset of an unverified span in the chunk (ordinary-kernel launch)
  DevBuf<uint32_t> ls_dc_at;      // DC-blocker state at the start of an unverified span (34 words, word-major)
  PinnedBuf<uint32_t> ls_hctrl;   // mirror + scratch
  uint64_t ls_spec_launches = 0, ls_fallback_launches = 0;
  bool saw_f32 = false;           // an f32 submit happened since create / reset(all): DC state may be non-integer -> generic kernel
  uint64_t lost_events = 0, lost_payloads = 0;
  uint64_t rollbacks = 0;          // option "rollbacks"
  same_derived derived;
  DevBuf<uint32_t> d_state;
  DevBuf<StreamBlob> d_blobs;
  DevBuf<same_event> d_events;
  DevBuf<same_event> d_sorted;           // arena events counting-sorted by (stream, seq) before read-back
  DevBuf<uint32_t> d_sort_ws;            // cnt[n+1] | start[n+1] | minseq[n] | bad[1]
  bool pend_sorted = false;              // pend_events is one device-sorted batch: drain copies it as it is
  int device_sort = 1;                   // option "device_sort": 0 = always sort on the host (diagnostic)
  DevBuf<uint8_t> d_payload;
  DevBuf<unsigned int> d_counters;
  PinnedBuf<unsigned int> h_counters;
  PinnedBuf<uint8_t> h_stage;            // staging for device <-> pageable host copies (STAGE_BYTES, used as two halves)
  Event stage_done[2];
  DevBuf<same_soft_symbol> d_trace;      // n_streams x trace_cap symbols
  DevBuf<uint32_t> d_ids;
  InputBuf in[2];
  int cur = 0;
  bool in_flight = false;
  std::vector<same_event> pend_events;
  std::vector<uint8_t> pend_payload;
  Event t_h2d0, t_h2d1, t_k0, t_k1, t_sw0, t_sw1;
  bool timed_h2d = false, timed_kernel = false;
  // portable stream state (same_state.cu): device staging of records, ids, validation result, timing of the last call
  DevBuf<uint8_t> d_xfer;
  DevBuf<uint32_t> d_xids;
  DevBuf<unsigned long long> d_xres;
  Event t_st[3];
  float st_kernel_ms = 0.0f, st_copy_ms = 0.0f;
  uint64_t launches = 0;
  std::string last_error;
};

namespace {

int fail(same_engine* e, int code, const std::string& msg) {
  if (e) e->last_error = msg;
  g_last_error = msg;
  return code;
}

#define CK(e, call)                                                                                     \
  do {                                                                                                  \
    cudaError_t _err = (call);                                                                          \
    if (_err != cudaSuccess)                                                                            \
      return fail((e), SAME_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_err));            \
  } while (0)

// The kernel parameters that point into the engine's buffers, set from their owners after any of them changed
void bind(same_engine* e) {
  SameParams& p = e->p;
  p.state32 = e->d_state; p.blobs = e->d_blobs; p.counters = e->d_counters;
  p.events = e->d_events; p.payload = e->d_payload;
  p.events_cap = (uint32_t)std::min<size_t>(e->d_events.size(), 0xffffffffu);
  p.payload_cap = (uint32_t)std::min<size_t>(e->d_payload.size(), 0xffffffffu);
  p.trace = e->d_trace; p.trace_cap = (uint32_t)(e->d_trace.size() / e->n_streams);
  e->tiles.d = e->tiles_d; e->tiles.dc_next = e->tiles_dc_next;
}

// Event arenas of exactly these sizes; the old ones stay in use unless all of the new ones could be allocated
int alloc_arenas(same_engine* e, size_t max_events, size_t max_payload) {
  DevBuf<same_event> events, sorted;
  DevBuf<uint8_t> payload;
  CK(e, events.grow(max_events));
  CK(e, sorted.grow(max_events));
  CK(e, payload.grow(max_payload));
  e->d_events.swap(events); e->d_sorted.swap(sorted); e->d_payload.swap(payload);
  bind(e);
  return SAME_OK;
}

static const size_t STAGE_BYTES = 2 * 48 * 32768;   // two halves of 32768 events (1.5 MiB each)

// device -> pinned staging -> take(slice, n) for each slice in order: two halves, so that the copy of one slice overlaps
// the host's use of the other
template <class Take>
int stage_out(same_engine* e, const uint8_t* src, size_t bytes, Take&& take) {
  const size_t half = STAGE_BYTES / 2;
  size_t done = 0, queued = 0, qn[2] = {0, 0};
  int qslot = 0, pslot = 0, inflight = 0;
  while (done < bytes) {
    while (inflight < 2 && queued < bytes) {   // keep both halves in flight
      const size_t n = std::min(half, bytes - queued);
      CK(e, cudaMemcpyAsync(e->h_stage + qslot * half, src + queued, n, cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaEventRecord(e->stage_done[qslot], e->compute));
      qn[qslot] = n; queued += n; qslot ^= 1; ++inflight;
    }
    CK(e, cudaEventSynchronize(e->stage_done[pslot]));
    take(e->h_stage + pslot * half, qn[pslot]);
    done += qn[pslot]; pslot ^= 1; --inflight;
  }
  return SAME_OK;
}

// Pull the events produced since the last collect from the device arenas into the host pending lists.
int collect(same_engine* e) {
  CK(e, cudaMemcpyAsync(e->h_counters, e->d_counters, 4 * sizeof(unsigned int), cudaMemcpyDeviceToHost, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  const size_t nev = e->h_counters[0], npay = e->h_counters[1];
  e->rollbacks += e->h_counters[3];
  const size_t events_cap = e->d_events.size(), payload_cap = e->d_payload.size();
  int rc = SAME_OK;
  if (nev > events_cap || e->h_counters[2] != 0) {
    // Events beyond the arena were dropped by the device; events whose payload did not fit were stored with
    // data_len 0 + SAME_EV_FLAG_PAYLOAD_LOST (same_transport.cuh:emit_event_impl), so everything handed to the caller
    // below stays self-consistent.  The stream state has advanced: what was dropped is lost, and counted.
    const uint64_t ev_lost = nev > events_cap ? nev - events_cap : 0;
    e->lost_events += ev_lost;
    e->lost_payloads += e->h_counters[2];
    char buf[256];
    snprintf(buf, sizeof buf, "event arena overflow since the last sync: %llu events dropped (capacity %zu), %u payloads dropped "
             "(capacity %zu bytes)", (unsigned long long)ev_lost, events_cap, e->h_counters[2], payload_cap);
    rc = fail(e, SAME_ERR_EVENT_OVERFLOW, buf);
  }
  const size_t cev = std::min(nev, events_cap), cpay = std::min(npay, payload_cap);
  // big single batches are put into (stream, occurrence) order on the device; the host sort in drain is the fallback
  const same_event* ev_src = e->d_events;
  bool dev_sorted = false;
  if (rc == SAME_OK && e->device_sort && cev >= 4096 && e->pend_events.empty() && cev <= 0xffffffffu) {
    uint32_t* cnt = e->d_sort_ws;
    uint32_t* start = cnt + e->n_streams + 1;
    uint32_t* minseq = start + e->n_streams + 1;
    uint32_t* bad = minseq + e->n_streams;
    CK(e, same_launch_evsort(e->d_events, (uint32_t)cev, e->n_streams, cnt, minseq, start, e->d_sorted, bad, e->compute));
    e->launches += 3;   // histogram, scan, scatter
    CK(e, cudaMemcpyAsync(e->h_counters, bad, sizeof(unsigned int), cudaMemcpyDeviceToHost, e->compute));
    CK(e, cudaStreamSynchronize(e->compute));
    if (e->h_counters[0] == 0) { ev_src = e->d_sorted; dev_sorted = true; }
  }
  e->pend_sorted = dev_sorted || (cev == 0 && e->pend_sorted);
  if (cev) {
    // appended slice by slice: the staging halves hold whole events
    const size_t base_ev = e->pend_events.size(), base_pay = e->pend_payload.size();
    e->pend_events.reserve(base_ev + cev);
    e->pend_payload.reserve(base_pay + cpay);
    int r = stage_out(e, reinterpret_cast<const uint8_t*>(ev_src), cev * sizeof(same_event), [e](const uint8_t* h, size_t n) {
      const same_event* ev = reinterpret_cast<const same_event*>(h);
      e->pend_events.insert(e->pend_events.end(), ev, ev + n / sizeof(same_event));
    });
    if (r) return r;
    r = stage_out(e, e->d_payload, cpay, [e](const uint8_t* h, size_t n) { e->pend_payload.insert(e->pend_payload.end(), h, h + n); });
    if (r) return r;
    for (size_t i = base_ev; i < base_ev + cev; ++i) {
      same_event& ev = e->pend_events[i];
      const uint32_t stored = ev.kind == SAME_EV_LINK_BURST ? std::min<uint32_t>(ev.data_len, SAME_BURST_CAP) : ev.data_len;
      if ((size_t)ev.data_offset + stored > cpay) {   // cannot happen with a sane device record: never hand out a bad offset
        ev.data_offset = 0; ev.data_len = 0; ev.flags |= SAME_EV_FLAG_PAYLOAD_LOST;
      }
      ev.data_offset += (uint32_t)base_pay;
    }
  }
  CK(e, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned int), e->compute));
  return rc;
}

// Drop the undrained events of streams ids[0..n) (nullptr: 0..n-1); their payload bytes stay until the next drain
void forget_events(same_engine* e, const uint32_t* ids, uint32_t n) {
  std::vector<char> hit(e->n_streams, 0);
  for (uint32_t i = 0; i < n; ++i) hit[ids ? ids[i] : i] = 1;
  e->pend_events.erase(std::remove_if(e->pend_events.begin(), e->pend_events.end(),
                                      [&](const same_event& ev) { return hit[ev.stream] != 0; }),
                       e->pend_events.end());
}

// Tile buffer of the split pipeline: n_pad streams x n_max samples of f32 (+ the 34-word DC state per stream).
int ensure_tiles(same_engine* e, uint32_t max_len) {
  const uint32_t n_max = (max_len + 31u) & ~31u;
  CK(e, e->tiles_d.grow((size_t)e->p.layout.n_pad * n_max));
  CK(e, e->tiles_dc_next.grow((size_t)34 * e->p.layout.n_pad));
  e->tiles.n_max = n_max;
  bind(e);
  return SAME_OK;
}

// ---- long-stream path: see same_long.cu ----
constexpr uint32_t kLongMinSamples = 65536;     // shorter chunks take the ordinary kernels
constexpr uint32_t kLongChunk = 1u << 24;       // samples per internal pass (bounds the scratch buffers: 16 B per sample)
constexpr uint32_t kLongSpan = 8192;            // samples per fallback launch while the AGC is locked (inside a burst)
constexpr uint32_t kLongSpanMax = 1u << 20;     // longest fallback span after verification stops in a row
constexpr uint32_t kLongMinPass = 1u << 16;     // shortest range of a speculative pass

int ensure_long(same_engine* e, size_t n) {
  CK(e, e->ls_d.grow(n + 64));
  CK(e, e->ls_y.grow(n + 128));
  CK(e, e->ls_g.grow(n + 64));
  CK(e, e->ls_soft.grow(n + 2 * 4096 + 64));   // + two tiles: the sequential kernel stages ahead
  CK(e, e->ls_gin.grow(n / 2048 + 8));
  CK(e, e->ls_ctrl.grow(4));
  CK(e, e->ls_hctrl.grow(8));
  CK(e, e->ls_off.grow(1));
  CK(e, e->ls_dc_at.grow((size_t)34 * e->p.layout.n_pad));
  CK(e, e->tiles_dc_next.grow((size_t)34 * e->p.layout.n_pad));
  bind(e);
  return SAME_OK;
}

// One stream, `len` device-resident s16 samples, on the compute stream.  Blocks the host (it steers the passes).
// A speculative pass covers [pos, pos + window).  Where the speculative AGC's hand-overs verify (loud noise, a gain
// pinned at a limit) the window doubles after every pass that consumed all of it, so a burst-free chunk takes one pass.
// Where they do not (quiet noise, DESIGN.md §4) a pass stops at its verified end: the window halves, and the samples
// after that end go to the ordinary pipelined kernel on the raw samples, in a span that doubles with every stop in a
// row (the DC-blocker state is first brought to the span's start by kernel A).  So no pass costs more than a constant
// times what it consumes plus what the pass before it consumed, and input that never verifies runs at the ordinary
// kernel's speed.  Bursts (AGC locked) go to the tile-fed single-warp kernel on A's output, kLongSpan at a time.
int run_long(same_engine* e, const int16_t* d_src, uint32_t len) {
  const SameLayout& L = e->p.layout;
  for (uint32_t base = 0; base < len; base += kLongChunk) {
    const uint32_t n = std::min(kLongChunk, len - base);
    int rc = ensure_long(e, n);
    if (rc) return rc;
    const int16_t* src = d_src + base;
    CK(e, same_long_launch_dc(&e->p, src, n, e->ls_d, e->tiles_dc_next, e->compute));
    e->launches += 1;
    // dc_at: the position the resident DC-blocker state belongs to (the state words are committed at the chunk's end)
    uint32_t pos = 0, window = n, unverified = 0, stops = 0, dc_at = 0;
    while (pos < n) {
      if (unverified) {   // the span after a verification stop: the ordinary kernel on the raw samples
        const uint32_t span = std::min(unverified, n - pos);
        if (dc_at < pos) {
          CK(e, same_long_launch_dc(&e->p, src + dc_at, pos - dc_at, e->ls_y, e->ls_dc_at, e->compute));
          CK(e, same_long_launch_commit_dc(&e->p, e->ls_dc_at, e->compute));
          e->launches += 2;
        }
        e->ls_hctrl[5] = span;
        *reinterpret_cast<unsigned long long*>(e->ls_hctrl + 6) = pos;
        CK(e, cudaMemcpyAsync(e->ls_ctrl + 3, e->ls_hctrl + 5, sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
        CK(e, cudaMemcpyAsync(e->ls_off, e->ls_hctrl + 6, sizeof(unsigned long long), cudaMemcpyHostToDevice, e->compute));
        CK(e, same_launch_rx(&e->p, &e->taps, &e->taps2, &e->taps_wide, PIPE, e->lanes_per_warp, src, 0, e->ls_off, e->ls_ctrl + 3, nullptr,
                             e->compute));
        e->launches += 1; e->ls_fallback_launches += 1;
        pos += span;
        dc_at = pos;
        unverified = 0;
        continue;
      }
      // is the AGC locked (inside a burst)?  then the samples are the ordinary kernel's, span by span
      CK(e, cudaMemcpyAsync(e->ls_hctrl + 4, e->d_state + (size_t)F_FLAGS * L.n_pad, sizeof(uint32_t), cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaStreamSynchronize(e->compute));
      if (e->ls_hctrl[4] & FLAG_AGC_LOCKED) {
        const uint32_t span = std::min(kLongSpan, n - pos);
        e->ls_hctrl[5] = span;
        CK(e, cudaMemcpyAsync(e->ls_ctrl + 3, e->ls_hctrl + 5, sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
        SameTiles t{e->ls_d + pos, e->tiles_dc_next, span, 1u, 0u};
        CK(e, same_launch_rx_tilefed(&e->p, &e->taps2, e->ls_ctrl + 3, &t, e->compute));
        e->launches += 1; e->ls_fallback_launches += 1;
        pos += span;
        continue;
      }
      const uint32_t end = pos + std::min(window, n - pos);
      CK(e, same_long_launch_speculative(&e->p, &e->taps2, e->ls_d, pos, end, e->ls_y, e->ls_g, e->ls_gin, e->ls_soft, e->ls_ctrl,
                                         e->compute));
      e->launches += 4; e->ls_spec_launches += 1;
      CK(e, cudaMemcpyAsync(e->ls_hctrl, e->ls_ctrl, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaStreamSynchronize(e->compute));
      const uint32_t reached = e->ls_hctrl[1], why = e->ls_hctrl[2];
      if (reached < pos || reached > end) return fail(e, SAME_ERR_CUDA, "long-stream pass reported an impossible position");
      if (reached == pos && why == 0u) return fail(e, SAME_ERR_CUDA, "long-stream pass made no progress");
      pos = reached;
      if (why != 0u) continue;    // the symbol stages locked the AGC or reset the timing loop: the next round decides
      if (reached == end) {       // all of the range verified
        window = (uint32_t)std::min<uint64_t>(2ull * window, n);
        stops = 0;
      } else {                    // verification stop: the hand-over at `reached` did not match
        window = std::max(kLongMinPass, window / 2u);
        unverified = std::min(kLongSpanMax, kLongSpan << std::min(stops, 7u));
        stops += 1;
      }
    }
    CK(e, same_long_launch_commit_dc(&e->p, e->tiles_dc_next, e->compute));
    e->launches += 1;
  }
  return SAME_OK;
}

// The receiver kernel an s16 submit launches:
//  * the generic kernel once f32 input reached the state (saw_f32): the DC-blocker state may hold non-integers, and
//    the fast kernels' DC blocker is an integer recursion;
//  * the generic kernel for any geometry but the 22050 Hz class (42 taps, DC length 16), the fast kernels' only one;
//  * option "kernel";
//  * else the policy for the 22050 Hz class (measured on B200, tables in profiles/README.md), by 32-stream blocks per SM:
//    * <= 1: five-warp pipelined kernel (producer / AGC / space filter / timing loop / symbol stages), the timing warp
//      on a scheduler of its own: the per-stream dependent chain is what bounds the run time, so it is cut into stages.
//    * <= 4: three-warp kernel (producer / look-ahead AGC / consumer): fewer instructions in total, still
//      latency-hiding across the co-resident blocks.
//    * <= 8: single-warp fast kernel (8 resident blocks per SM: the whole batch is one wave; fewest instructions).
//    * more: single-warp look-ahead kernel (16 resident warps per SM, no d ring): the issue-bound regime.
//    20 s streams, ms per launch, pipelined / three-warp / single-warp / look-ahead: 4096 streams 24.0 / 24.9 / 41.6 / -;
//    8192: 36.8 / 29.1 / 43.3 / 66; 16384: 74.6 / 40.0 / 43.9 / 70; 32768: - / - / 57.7 / 81; 49152: - / - / 109 / 83;
//    65536: 228 / 158 / 116 / 97.
// Option "lanes_per_warp" spreads streams over more, lane-sparse warps (diagnostic).  No environment variable is read
// here: same_engine_set_option is the only override.
Kernel rx_kernel(const same_engine* e) {
  if (e->saw_f32 || e->p.ntaps != 42 || e->p.dc_len != 16) return GENERIC;
  if (e->kernel_override != POLICY) return e->kernel_override;
  const uint32_t blocks32 = (e->n_streams + 31u) / 32u, sms = (uint32_t)e->sm_count;
  return blocks32 <= sms ? PIPE : blocks32 <= 4u * sms ? THREE : blocks32 <= 8u * sms ? SINGLE : LOOKAHEAD;
}

struct Submit2D { uint64_t row_stride = 0, col_start = 0, dpitch = 0; uint32_t n_cols = 0; bool on = false; };

// sample_fmt: 0 = int16, 1 = float32
int submit_common(same_engine* e, const void* host_samples, const void* dev_samples, int sample_fmt, uint64_t total,
                  const uint64_t* offsets, const uint32_t* lengths, bool zeros, Submit2D two_d = Submit2D()) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  std::vector<uint64_t> off2d;
  std::vector<uint32_t> len2d;
  if (two_d.on) {
    if (!host_samples) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
    if (two_d.col_start + two_d.n_cols > two_d.row_stride) return fail(e, SAME_ERR_INVALID_ARG, "column range exceeds row_stride");
    // device rows are packed at a pitch that is a multiple of 8 samples, so that every row starts 16-byte aligned and
    // the fast kernels keep their 16-byte vector loads whatever n_cols is
    two_d.dpitch = ((uint64_t)two_d.n_cols + 7u) & ~(uint64_t)7u;
    off2d.resize(e->n_streams); len2d.assign(e->n_streams, two_d.n_cols);
    for (uint32_t i = 0; i < e->n_streams; ++i) off2d[i] = (uint64_t)i * two_d.dpitch;
    offsets = off2d.data(); lengths = len2d.data();
    total = (uint64_t)e->n_streams * two_d.dpitch;
  }
  if (!lengths || (!zeros && (!offsets || (!host_samples && !dev_samples && total))))
    return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  if (two_d.on && two_d.n_cols > (1u << 30)) return fail(e, SAME_ERR_INVALID_ARG, "chunk longer than 2^30 samples");
  CK(e, cudaSetDevice(e->device));
  if (!zeros)
    for (uint32_t i = 0; i < e->n_streams; ++i)
      if (lengths[i] && offsets[i] + lengths[i] > total)
        return fail(e, SAME_ERR_INVALID_ARG, "stream " + std::to_string(i) + ": offset+length exceeds total_samples");
  for (uint32_t i = 0; i < e->n_streams; ++i)
    if (lengths[i] > (1u << 30)) return fail(e, SAME_ERR_INVALID_ARG, "chunk longer than 2^30 samples");

  InputBuf& b = e->in[e->cur];
  e->cur ^= 1;
  // the copy stream may only overwrite this buffer after the kernel that last read it has finished
  if (b.used) CK(e, cudaStreamWaitEvent(e->copy, b.consumed, 0));
  e->timed_h2d = false;
  const void* d_src = nullptr;
  const size_t ssz = sample_fmt == 1 ? sizeof(float) : sizeof(int16_t);
  if (sample_fmt == 1) e->saw_f32 = true;
  if (!zeros) {
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "offset type");
    CK(e, cudaMemcpyAsync(b.d_off, offsets, e->n_streams * sizeof(uint64_t), cudaMemcpyHostToDevice, e->copy));
  }
  CK(e, cudaMemcpyAsync(b.d_len, lengths, e->n_streams * sizeof(uint32_t), cudaMemcpyHostToDevice, e->copy));
  if (!zeros && host_samples) {
    CK(e, b.d.grow(total * ssz, total * ssz / 8 + 8192));
    CK(e, cudaEventRecord(e->t_h2d0, e->copy));
    if (total && two_d.on)
      CK(e, cudaMemcpy2DAsync(b.d, (size_t)two_d.dpitch * ssz, static_cast<const uint8_t*>(host_samples) + two_d.col_start * ssz,
                              (size_t)two_d.row_stride * ssz, (size_t)two_d.n_cols * ssz,
                              e->n_streams, cudaMemcpyHostToDevice, e->copy));
    else if (total)
      CK(e, cudaMemcpyAsync(b.d, host_samples, total * ssz, cudaMemcpyHostToDevice, e->copy));
    CK(e, cudaEventRecord(e->t_h2d1, e->copy));
    e->timed_h2d = true;
    d_src = b.d;
  } else if (!zeros) {
    d_src = dev_samples;
  }
  CK(e, cudaEventRecord(b.copied, e->copy));
  CK(e, cudaStreamWaitEvent(e->compute, b.copied, 0));
  CK(e, cudaEventRecord(e->t_k0, e->compute));
  Kernel kernel = rx_kernel(e);
  // one stream, a long chunk: the long-stream path (time-parallel DC / AGC / matched filters, sequential timing loop)
  const bool long_path = e->long_stream && e->n_streams == 1 && d_src && e->kernel_override == POLICY && kernel != GENERIC &&
                         lengths[0] >= kLongMinSamples;
  // the split pipeline's front end needs real samples: a zeros submit has none and takes the fused single-warp kernel
  // (the resident state is the same)
  if (kernel == SPLIT && !d_src) kernel = SINGLE;
  if (long_path) {
    int rc = run_long(e, static_cast<const int16_t*>(d_src) + offsets[0], lengths[0]);
    if (rc) return rc;
  } else {
    if (kernel == SPLIT) {   // a tile buffer for the longest chunk
      uint32_t max_len = 0;
      for (uint32_t i = 0; i < e->n_streams; ++i) max_len = std::max(max_len, lengths[i]);
      int rc = ensure_tiles(e, max_len);
      if (rc) return rc;
      e->launches += 1;   // the front-end kernel
    }
    CK(e, same_launch_rx(&e->p, &e->taps, &e->taps2, &e->taps_wide, kernel, e->lanes_per_warp, d_src, sample_fmt, b.d_off, b.d_len,
                         &e->tiles, e->compute));
    e->launches += 1;
  }
  CK(e, cudaEventRecord(e->t_k1, e->compute));
  CK(e, cudaEventRecord(b.consumed, e->compute));
  b.used = true;
  e->timed_kernel = true;
  e->in_flight = true;
  return SAME_OK;
}

}  // namespace

extern "C" {

uint32_t same_abi_version(void) { return SAME_ABI_VERSION; }
const char* same_last_error(void) { return g_last_error.c_str(); }
const char* same_engine_last_error(const same_engine* e) { return e ? e->last_error.c_str() : g_last_error.c_str(); }

void same_config_default(same_config* c, uint32_t input_rate) {  // builder.rs:50-67, 369-376
  if (!c) return;
  c->input_rate = input_rate;
  c->dc_blocker_len = 0.38f;
  c->agc_bandwidth = 0.01f;
  c->agc_gain_min = 0.0f; c->agc_gain_max = 1.0e6f;
  c->timing_bw_unlocked = 0.125f; c->timing_bw_locked = 0.05f;
  c->timing_max_deviation = 0.01f;
  c->squelch_power_open = 0.10f; c->squelch_power_close = 0.05f;
  c->squelch_bandwidth = 0.125f;
  c->preamble_max_errors = 2;
  c->eq_enabled = 1; c->eq_nff = 6; c->eq_nfb = 4;
  c->eq_relaxation = 0.05f; c->eq_regularization = 1.0e-6f;
  c->frame_prefix_max_errors = 2; c->frame_max_invalid_bytes = 5;
}

void same_config_samedec(same_config* c, uint32_t input_rate) {  // crates/samedec/src/main.rs:29-37
  if (!c) return;
  same_config_default(c, input_rate);
  c->agc_gain_min = 1.0f / (float)INT16_MAX;
  c->agc_gain_max = 1.0f / 200.0f;
}

void same_config_sanitize(same_config* c) {  // the with_* setters, builder.rs:95-279, 393-425
  if (!c) return;
  c->dc_blocker_len = fmaxf(0.0f, c->dc_blocker_len);
  c->agc_bandwidth = rclampf(c->agc_bandwidth, 0.0f, 1.0f);
  c->timing_bw_unlocked = rclampf(c->timing_bw_unlocked, 0.0f, 1.0f);
  c->timing_bw_locked = rclampf(c->timing_bw_locked, 0.0f, c->timing_bw_unlocked);
  c->timing_max_deviation = rclampf(c->timing_max_deviation, 0.0f, 0.5f);
  {
    float open = c->squelch_power_open, close = c->squelch_power_close;
    c->squelch_power_open = rclampf(open, 0.0f, 1.0f);
    c->squelch_power_close = fminf(close, open);
  }
  c->frame_prefix_max_errors = std::min<uint32_t>(c->frame_prefix_max_errors, 7u);
  c->eq_nff = std::max<uint32_t>(c->eq_nff, 1u);
  c->eq_nfb = std::min<uint32_t>(std::max<uint32_t>(c->eq_nfb, 1u), c->eq_nff);
  c->eq_relaxation = rclampf(c->eq_relaxation, 0.0f, 1.0f);
  c->eq_regularization = rclampf(c->eq_regularization, 0.0f, 3.40282347e+38f);
}

int same_engine_create(const same_config* cfg_in, int device, uint32_t n_streams, same_engine** out) {
  if (!cfg_in || !out) return fail(nullptr, SAME_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (n_streams == 0 || n_streams > (1u << 24)) return fail(nullptr, SAME_ERR_INVALID_ARG, "n_streams out of range");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, SAME_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(nullptr, SAME_ERR_NO_DEVICE, "device index out of range");

  same_config cfg = *cfg_in;
  same_config_sanitize(&cfg);
  if (cfg.input_rate == 0) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "input_rate must be > 0");
  if (!(cfg.agc_gain_min <= cfg.agc_gain_max))  // f32::clamp panics when min > max or either is NaN (agc.rs:75)
    return fail(nullptr, SAME_ERR_INVALID_CONFIG, "agc_gain_min must be <= agc_gain_max");

  // ---- SameReceiver::from(&builder)  receiver.rs:502-560 ----
  const float rate_f = (float)cfg.input_rate;
  const float sps = same_samples_per_symbol(cfg.input_rate);                  // waveform.rs:29-31
  const size_t dc_len = same_f32_as_usize(cfg.dc_blocker_len * sps);          // receiver.rs:509
  const size_t ntaps = same_ntaps(cfg.input_rate);                            // waveform.rs:40
  if (dc_len == 0) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "DC blocker length is 0 samples (MovingAverage::new asserts len > 0, dcblock.rs:74)");
  if (dc_len > SAME_MAX_DC)
    return fail(nullptr, SAME_ERR_INVALID_CONFIG, "DC blocker of " + std::to_string(dc_len) + " samples is longer than the engine limit of " +
                                                      std::to_string(SAME_MAX_DC) + " samples");
  if (ntaps == 0 || ntaps > SAME_MAX_TAPS) {
    uint32_t lo, hi;
    rate_range(SAME_MAX_TAPS, &lo, &hi);
    return fail(nullptr, SAME_ERR_INVALID_CONFIG, "matched filter length outside 1.." + std::to_string(SAME_MAX_TAPS) + " taps (input_rate " +
                                                      std::to_string(lo) + ".." + std::to_string(hi) + " Hz)");
  }
  uint32_t nff = cfg.eq_enabled ? cfg.eq_nff : 1u, nfb = cfg.eq_enabled ? cfg.eq_nfb : 1u;   // disabled_equalizer() receiver.rs:585-590
  float relax = cfg.eq_enabled ? cfg.eq_relaxation : 0.0f;
  float regul = cfg.eq_enabled ? cfg.eq_regularization : 1.0e-6f;
  if (nff > SAME_MAX_EQ || nfb > SAME_MAX_EQ) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "equalizer order beyond the engine limit of 16 taps per arm");

  std::unique_ptr<same_engine, void (*)(same_engine*)> e(new same_engine(), same_engine_destroy);
  e->cfg = cfg; e->device = device; e->n_streams = n_streams;
  SameParams& p = e->p;
  memset(&p, 0, sizeof p);
  memset(&e->taps_wide, 0, sizeof e->taps_wide);
  memset(&e->taps, 0, sizeof e->taps);
  p.n_streams = n_streams; p.input_rate = cfg.input_rate;
  p.dc_len = (uint32_t)dc_len;
  p.dc_inv_len = 1.0f / (float)dc_len;                                        // dcblock.rs:77
  p.dc_gate = dc_len > 1 ? 1.0f : 0.0f;                                       // dcblock.rs:48
  p.agc_bw = rclampf(cfg.agc_bandwidth * sps / rate_f, 0.0f, 1.0f);           // receiver.rs:511, agc.rs:51
  p.agc_min = cfg.agc_gain_min; p.agc_max = cfg.agc_gain_max;
  p.agc_gain0 = fminf(1.0f, cfg.agc_gain_min);                                // agc.rs:55
  p.ntaps = (uint32_t)ntaps;
  {
    std::vector<float> mre(p.ntaps), mim(p.ntaps), sre(p.ntaps), sim(p.ntaps);
    cisoid_taps(p.ntaps, kMarkHz / rate_f, mre.data(), mim.data());           // waveform.rs:41-42
    cisoid_taps(p.ntaps, kSpaceHz / rate_f, sre.data(), sim.data());
    for (uint32_t i = 0; i < p.ntaps; ++i) e->taps_wide.t[i] = make_float4(mre[i], mim[i], sre[i], sim[i]);
  }
  for (uint32_t i = 0; i < p.ntaps && i < SAME_GENERIC_TAPS; ++i) {
    const float4 t = e->taps_wide.t[i];
    e->taps.mark_re[i] = t.x; e->taps.mark_im[i] = t.y; e->taps.space_re[i] = t.z; e->taps.space_im[i] = t.w;
  }
  memset(&e->taps2, 0, sizeof e->taps2);
  for (uint32_t i = 0; i < p.ntaps && i < 64; ++i) {
    e->taps2.mark[i] = make_float2(e->taps.mark_re[i], e->taps.mark_im[i]);
    e->taps2.space[i] = make_float2(e->taps.space_re[i], e->taps.space_im[i]);
  }
  p.f_one = 1.0f; p.f_negzero = -0.0f;
  {
    int sms = 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
    e->sm_count = sms;   // for the kernel policy (rx_kernel)
  }
  p.spt = sps / 2.0f;                                                         // symsync.rs:146
  {
    float dev = sps * rclampf(cfg.timing_max_deviation, 0.0f, 0.5f);          // symsync.rs:147
    p.pmin = p.spt - dev; p.pmax = p.spt + dev;
  }
  loop_alphabeta(cfg.timing_bw_unlocked, p.alpha_u, p.beta_u);
  loop_alphabeta(cfg.timing_bw_locked, p.alpha_l, p.beta_l);
  p.sq_sync_word = 0xabababab;                                                // waveform.rs:26
  p.sq_max_err = cfg.preamble_max_errors;
  p.sq_open = cfg.squelch_power_open;
  p.sq_close = fminf(cfg.squelch_power_close, cfg.squelch_power_open);        // codesquelch.rs:199
  p.sq_bw = rclampf(cfg.squelch_bandwidth, 0.0f, 1.0f);                       // codesquelch.rs:468
  p.eq_nff = nff; p.eq_nfb = nfb; p.eq_relax = relax; p.eq_regul = regul;
  p.fr_max_prefix_err = cfg.frame_prefix_max_errors; p.fr_max_invalid = cfg.frame_max_invalid_bytes;
  {
    float ib = (1.05f * kBaudHz) + 17.0f * 8.0f;                              // assembler.rs:85
    p.interburst_symbols = (unsigned long long)ib;
    p.history_symbols = 2ull * (p.interburst_symbols + 8ull * SAME_MAX_MESSAGE_LENGTH);  // assembler.rs:92-93
    p.force_eom_samples = 135ull * (unsigned long long)cfg.input_rate;        // receiver.rs:496, 321-324
  }
  SameLayout& L = p.layout;
  L.n_pad = (n_streams + 31u) & ~31u;
  uint32_t w = F_NUM_SCALARS;
  L.dc_ff = w; w += p.dc_len;
  L.dc_fb = w; w += p.dc_len;
  L.win = w; w += p.ntaps;
  L.sqh = w; w += SAME_SQ_HIST;
  L.eq_ffc = w; w += nff;
  L.eq_fbc = w; w += nfb;
  L.eq_ffw = w; w += nff;
  L.eq_fbw = w; w += nfb;
  L.n_words = w;

  e->derived.sps = sps; e->derived.agc_bw = p.agc_bw; e->derived.agc_gain0 = p.agc_gain0;
  e->derived.samples_per_ted = p.spt; e->derived.period_min = p.pmin; e->derived.period_max = p.pmax;
  e->derived.alpha_unlocked = p.alpha_u; e->derived.beta_unlocked = p.beta_u;
  e->derived.alpha_locked = p.alpha_l; e->derived.beta_locked = p.beta_l;
  e->derived.dc_len = p.dc_len; e->derived.ntaps = p.ntaps;

  CK(nullptr, cudaSetDevice(device));
  CK(nullptr, e->compute.create());
  CK(nullptr, e->copy.create());
  CK(nullptr, e->d_state.grow((size_t)L.n_words * L.n_pad));
  CK(nullptr, e->d_blobs.grow(n_streams));
  CK(nullptr, cudaMemsetAsync(e->d_blobs, 0, (size_t)n_streams * sizeof(StreamBlob), e->compute));
  CK(nullptr, e->d_counters.grow(4));
  CK(nullptr, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned int), e->compute));
  CK(nullptr, e->d_sort_ws.grow(3 * (size_t)n_streams + 3));
  CK(nullptr, e->h_counters.grow(4));
  CK(nullptr, e->h_stage.grow(STAGE_BYTES));
  for (Event& ev : e->stage_done) CK(nullptr, ev.create(cudaEventDisableTiming));
  for (InputBuf& b : e->in) {
    CK(nullptr, b.d_off.grow(n_streams));
    CK(nullptr, b.d_len.grow(n_streams));
    CK(nullptr, b.copied.create(cudaEventDisableTiming));
    CK(nullptr, b.consumed.create(cudaEventDisableTiming));
  }
  for (Event* ev : {&e->t_h2d0, &e->t_h2d1, &e->t_k0, &e->t_k1, &e->t_sw0, &e->t_sw1}) CK(nullptr, ev->create());
  for (Event& ev : e->t_st) CK(nullptr, ev.create());
  const int rc = alloc_arenas(e.get(), std::max<size_t>(65536, (size_t)n_streams * 64),
                              std::max<size_t>(4u << 20, (size_t)n_streams * 4096));   // binds the kernel parameters
  if (rc) return rc;
  CK(nullptr, same_launch_init(&e->p, nullptr, n_streams, 0, e->compute));
  CK(nullptr, cudaStreamSynchronize(e->compute));
  *out = e.release();
  return SAME_OK;
}

// Everything the engine owns is released by its members' destructors, once the work queued on its streams is done.
void same_engine_destroy(same_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->compute) cudaStreamSynchronize(e->compute);
  if (e->copy) cudaStreamSynchronize(e->copy);
  delete e;
}

uint32_t same_engine_num_streams(const same_engine* e) { return e ? e->n_streams : 0; }
uint32_t same_engine_input_rate(const same_engine* e) { return e ? e->cfg.input_rate : 0; }
uint64_t same_engine_launch_count(const same_engine* e) { return e ? e->launches : 0; }
void* same_engine_cuda_stream(same_engine* e) { return e ? (void*)e->compute : nullptr; }

int same_engine_sync(same_engine* e) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  CK(e, cudaSetDevice(e->device));
  CK(e, cudaStreamSynchronize(e->copy));
  CK(e, cudaStreamSynchronize(e->compute));
  if (!e->in_flight) return SAME_OK;
  e->in_flight = false;
  return collect(e);
}

int same_engine_input_sample_counters(same_engine* e, uint64_t* out) {
  if (!e || !out) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  const SameLayout& L = e->p.layout;
  std::vector<uint32_t> lo(e->n_streams), hi(e->n_streams);
  CK(e, cudaMemcpy(lo.data(), e->d_state + (size_t)F_N_LO * L.n_pad, e->n_streams * 4, cudaMemcpyDeviceToHost));
  CK(e, cudaMemcpy(hi.data(), e->d_state + (size_t)F_N_HI * L.n_pad, e->n_streams * 4, cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < e->n_streams; ++i) out[i] = ((uint64_t)hi[i] << 32) | lo[i];
  return SAME_OK;
}

int same_engine_reset(same_engine* e, const uint32_t* ids, uint32_t n) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  if (!ids) {
    CK(e, same_launch_init(&e->p, nullptr, e->n_streams, 1, e->compute));
    e->launches += 1;
    // SameReceiver::reset clears the event queue (receiver.rs:194)
    e->pend_events.clear(); e->pend_payload.clear();
    e->saw_f32 = false;   // every DC-blocker window is zero again
  } else {
    for (uint32_t i = 0; i < n; ++i)
      if (ids[i] >= e->n_streams) return fail(e, SAME_ERR_INVALID_ARG, "stream id out of range");
    CK(e, e->d_ids.grow(n));
    CK(e, cudaMemcpyAsync(e->d_ids, ids, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
    CK(e, same_launch_init(&e->p, e->d_ids, n, 1, e->compute));
    e->launches += 1;
    forget_events(e, ids, n);
  }
  CK(e, cudaStreamSynchronize(e->compute));
  return SAME_OK;
}

struct same_snapshot {
  int device = 0;
  uint32_t n_streams = 0;
  bool saw_f32 = false;   // the DC-blocker state may be non-integer: restore must keep the engine on the generic kernel
  DevBuf<uint32_t> d_state;
  DevBuf<StreamBlob> d_blobs;
};

int same_engine_snapshot(same_engine* e, same_snapshot** out) {
  if (!e || !out) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  std::unique_ptr<same_snapshot> s(new same_snapshot());
  s->device = e->device; s->n_streams = e->n_streams;
  s->saw_f32 = e->saw_f32;
  cudaError_t err = s->d_state.grow(e->d_state.size());
  if (err == cudaSuccess) err = s->d_blobs.grow(e->d_blobs.size());
  if (err == cudaSuccess)
    err = cudaMemcpyAsync(s->d_state, e->d_state, e->d_state.size() * sizeof(uint32_t), cudaMemcpyDeviceToDevice, e->compute);
  if (err == cudaSuccess)
    err = cudaMemcpyAsync(s->d_blobs, e->d_blobs, e->d_blobs.size() * sizeof(StreamBlob), cudaMemcpyDeviceToDevice, e->compute);
  if (err == cudaSuccess) err = cudaStreamSynchronize(e->compute);
  if (err != cudaSuccess) return fail(e, SAME_ERR_CUDA, std::string("snapshot: ") + cudaGetErrorString(err));
  *out = s.release();
  return SAME_OK;
}

int same_engine_restore(same_engine* e, const same_snapshot* s) {
  if (!e || !s) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  if (s->device != e->device || s->n_streams != e->n_streams || s->d_state.size() != e->d_state.size())
    return fail(e, SAME_ERR_INVALID_ARG, "snapshot belongs to a different engine shape");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  CK(e, cudaMemcpyAsync(e->d_state, s->d_state, e->d_state.size() * sizeof(uint32_t), cudaMemcpyDeviceToDevice, e->compute));
  CK(e, cudaMemcpyAsync(e->d_blobs, s->d_blobs, e->d_blobs.size() * sizeof(StreamBlob), cudaMemcpyDeviceToDevice, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  e->pend_events.clear(); e->pend_payload.clear();
  e->saw_f32 = s->saw_f32;
  return SAME_OK;
}

void same_snapshot_free(same_snapshot* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  delete s;
}

int same_engine_set_event_capacity(same_engine* e, size_t max_events, size_t max_payload_bytes) {
  if (!e || max_events == 0 || max_payload_bytes == 0) return fail(e, SAME_ERR_INVALID_ARG, "bad capacity");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  return alloc_arenas(e, max_events, max_payload_bytes);
}

int same_engine_submit_s16(same_engine* e, const int16_t* samples, uint64_t total_samples, const uint64_t* offsets,
                           const uint32_t* lengths) {
  return submit_common(e, samples, nullptr, 0, total_samples, offsets, lengths, false);
}

int same_engine_submit_f32(same_engine* e, const float* samples, uint64_t total_samples, const uint64_t* offsets,
                           const uint32_t* lengths) {
  return submit_common(e, samples, nullptr, 1, total_samples, offsets, lengths, false);
}

int same_engine_submit_f32_device(same_engine* e, const float* d_samples, uint64_t total_samples,
                                  const uint64_t* offsets, const uint32_t* lengths) {
  return submit_common(e, nullptr, d_samples, 1, total_samples, offsets, lengths, false);
}

int same_engine_lost_events(same_engine* e, uint64_t* events_lost, uint64_t* payloads_lost) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (e->in_flight) { int rc = same_engine_sync(e); if (rc && rc != SAME_ERR_EVENT_OVERFLOW) return rc; }
  if (events_lost) *events_lost = e->lost_events;
  if (payloads_lost) *payloads_lost = e->lost_payloads;
  return SAME_OK;
}

int same_engine_submit_s16_2d(same_engine* e, const int16_t* samples, uint64_t row_stride, uint64_t col_start,
                              uint32_t n_cols) {
  Submit2D t; t.row_stride = row_stride; t.col_start = col_start; t.n_cols = n_cols; t.on = true;
  return submit_common(e, samples, nullptr, 0, 0, nullptr, nullptr, false, t);
}

int same_engine_submit_s16_device(same_engine* e, const int16_t* d_samples, uint64_t total_samples,
                                  const uint64_t* offsets, const uint32_t* lengths) {
  return submit_common(e, nullptr, d_samples, 0, total_samples, offsets, lengths, false);
}

int same_engine_submit_zeros(same_engine* e, const uint32_t* lengths) {
  return submit_common(e, nullptr, nullptr, 0, 0, nullptr, lengths, true);
}

int same_engine_pending(same_engine* e, size_t* n_events, size_t* n_payload_bytes) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (e->in_flight) { int rc = same_engine_sync(e); if (rc) return rc; }
  if (n_events) *n_events = e->pend_events.size();
  if (n_payload_bytes) *n_payload_bytes = e->pend_payload.size();
  return SAME_OK;
}

int same_engine_drain_events(same_engine* e, same_event* events, size_t events_cap, size_t* n_events, uint8_t* payload,
                             size_t payload_cap, size_t* n_payload) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (e->in_flight) { int rc = same_engine_sync(e); if (rc) return rc; }
  const size_t nev = e->pend_events.size(), npay = e->pend_payload.size();
  if (n_events) *n_events = nev;
  if (n_payload) *n_payload = npay;
  if (nev > events_cap || npay > payload_cap || (nev && !events) || (npay && !payload))
    return fail(e, SAME_ERR_INVALID_ARG, "drain buffers too small");
  // per-stream order of occurrence, as iter_events yields them (receiver.rs:238-240, 267-269): counting sort by
  // stream straight into the caller's buffer, then order each stream's few events by sequence number
  if (nev && e->pend_sorted) {
    memcpy(events, e->pend_events.data(), nev * sizeof(same_event));   // already in (stream, occurrence) order
  } else if (nev) {
    std::vector<uint32_t> start(e->n_streams + 1, 0);
    for (const same_event& ev : e->pend_events) start[std::min(ev.stream, e->n_streams - 1) + 1] += 1;
    for (uint32_t i = 0; i < e->n_streams; ++i) start[i + 1] += start[i];
    std::vector<uint32_t> fill(start.begin(), start.end() - 1);
    for (const same_event& ev : e->pend_events) events[fill[std::min(ev.stream, e->n_streams - 1)]++] = ev;
    for (uint32_t i = 0; i < e->n_streams; ++i) {
      same_event* a = events + start[i];
      const uint32_t m = start[i + 1] - start[i];
      for (uint32_t j = 1; j < m; ++j) {   // insertion sort: nearly sorted, a handful of events per stream
        same_event t = a[j];
        uint32_t k = j;
        while (k > 0 && a[k - 1].seq > t.seq) { a[k] = a[k - 1]; --k; }
        a[k] = t;
      }
    }
  }
  if (npay) memcpy(payload, e->pend_payload.data(), npay);
  e->pend_events.clear(); e->pend_payload.clear();
  e->pend_sorted = false;
  return SAME_OK;
}

int same_engine_enable_soft_trace(same_engine* e, uint32_t cap_per_stream) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  DevBuf<same_soft_symbol> trace;   // exactly cap_per_stream symbols per stream (none: tracing off)
  CK(e, trace.grow((size_t)e->n_streams * cap_per_stream));
  const SameLayout& L = e->p.layout;
  CK(e, cudaMemset(e->d_state + (size_t)F_TRACE_N * L.n_pad, 0, (size_t)L.n_pad * 4));
  e->d_trace.swap(trace);
  bind(e);
  return SAME_OK;
}

int same_engine_read_soft_trace(same_engine* e, uint32_t stream, same_soft_symbol* out, size_t cap, size_t* n) {
  if (!e || !n || stream >= e->n_streams) return fail(e, SAME_ERR_INVALID_ARG, "bad argument");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  *n = 0;
  if (!e->d_trace) return SAME_OK;
  const SameLayout& L = e->p.layout;
  uint32_t fill = 0;
  CK(e, cudaMemcpy(&fill, e->d_state + (size_t)F_TRACE_N * L.n_pad + stream, 4, cudaMemcpyDeviceToHost));
  *n = fill;
  if (out) {
    size_t c = std::min<size_t>(fill, cap);
    if (c) CK(e, cudaMemcpy(out, e->d_trace + (size_t)stream * e->p.trace_cap, c * sizeof(same_soft_symbol), cudaMemcpyDeviceToHost));
    // reading rewinds this stream's trace
    uint32_t zero = 0;
    CK(e, cudaMemcpy(e->d_state + (size_t)F_TRACE_N * L.n_pad + stream, &zero, 4, cudaMemcpyHostToDevice));
  }
  return SAME_OK;
}

int same_engine_set_option(same_engine* e, const char* key, int value) {
  if (!e || !key) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  if (strcmp(key, "kernel") == 0 || strcmp(key, "force_generic") == 0) {
    if (value < 0 || value > 6) return fail(e, SAME_ERR_INVALID_ARG, "kernel must be 0 (policy), 1 generic, 2 single-warp, 3 pipelined, 4 three-warp, 5 split (front end + tile-fed) or 6 look-ahead single-warp");
    e->kernel_override = (Kernel)value;
    return SAME_OK;
  }

  if (strcmp(key, "device_sort") == 0) { e->device_sort = value != 0; return SAME_OK; }
  if (strcmp(key, "long_stream") == 0) { e->long_stream = value != 0; return SAME_OK; }
  if (strcmp(key, "lanes_per_warp") == 0) {
    if (value < 1 || value > 32) return fail(e, SAME_ERR_INVALID_ARG, "lanes_per_warp must be in 1..32");
    e->lanes_per_warp = (uint32_t)value;
    return SAME_OK;
  }
  return fail(e, SAME_ERR_INVALID_ARG, std::string("unknown option ") + key);
}

int same_engine_get_option(same_engine* e, const char* key, int* value) {
  if (!e || !key || !value) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  if (strcmp(key, "kernel") == 0 || strcmp(key, "force_generic") == 0) { *value = e->kernel_override; return SAME_OK; }
  if (strcmp(key, "device_sort") == 0) { *value = e->device_sort; return SAME_OK; }
  if (strcmp(key, "long_stream") == 0) { *value = e->long_stream; return SAME_OK; }
  if (strcmp(key, "long_stream_passes") == 0) { *value = (int)std::min<uint64_t>(e->ls_spec_launches, 0x7fffffff); return SAME_OK; }
  if (strcmp(key, "long_stream_fallback_spans") == 0) { *value = (int)std::min<uint64_t>(e->ls_fallback_launches, 0x7fffffff); return SAME_OK; }
  if (strcmp(key, "lanes_per_warp") == 0) { *value = (int)e->lanes_per_warp; return SAME_OK; }
  if (strcmp(key, "state_kernel_us") == 0) { *value = (int)std::min(e->st_kernel_ms * 1000.0f, 2.0e9f); return SAME_OK; }
  if (strcmp(key, "state_copy_us") == 0) { *value = (int)std::min(e->st_copy_ms * 1000.0f, 2.0e9f); return SAME_OK; }
  if (strcmp(key, "kernel_selected") == 0) { *value = rx_kernel(e); return SAME_OK; }
  if (strcmp(key, "resident_blocks_per_sm") == 0) {
    CK(e, cudaSetDevice(e->device));
    CK(e, same_rx_resident_blocks(&e->p, rx_kernel(e), value));
    return SAME_OK;
  }
  if (strcmp(key, "rollbacks") == 0) { *value = (int)std::min<uint64_t>(e->rollbacks, 0x7fffffff); return SAME_OK; }
  return fail(e, SAME_ERR_INVALID_ARG, std::string("unknown option ") + key);
}

int same_engine_frontend_probe(same_engine* e, const int16_t* d_samples, uint64_t total_samples, const uint64_t* offsets,
                               const uint32_t* lengths, int reps, float* ms_per_launch) {
  if (!e || !d_samples || !offsets || !lengths || !ms_per_launch || reps < 1) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  if (e->p.ntaps != 42 || e->p.dc_len != 16) return fail(e, SAME_ERR_INVALID_CONFIG, "the front-end kernel is the 22050 Hz class (DC length 16)");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  uint32_t max_len = 0;
  for (uint32_t i = 0; i < e->n_streams; ++i) {
    if (lengths[i] && offsets[i] + lengths[i] > total_samples) return fail(e, SAME_ERR_INVALID_ARG, "offset+length exceeds total_samples");
    max_len = std::max(max_len, lengths[i]);
  }
  rc = ensure_tiles(e, max_len);
  if (rc) return rc;
  InputBuf& b = e->in[0];
  CK(e, cudaMemcpyAsync(b.d_off, offsets, e->n_streams * sizeof(uint64_t), cudaMemcpyHostToDevice, e->compute));
  CK(e, cudaMemcpyAsync(b.d_len, lengths, e->n_streams * sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
  CK(e, same_launch_frontend(&e->p, d_samples, b.d_off, b.d_len, &e->tiles, e->compute));   // warm-up
  CK(e, cudaEventRecord(e->t_k0, e->compute));
  for (int i = 0; i < reps; ++i) CK(e, same_launch_frontend(&e->p, d_samples, b.d_off, b.d_len, &e->tiles, e->compute));
  CK(e, cudaEventRecord(e->t_k1, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  float ms = 0.0f;
  CK(e, cudaEventElapsedTime(&ms, e->t_k0, e->t_k1));
  *ms_per_launch = ms / (float)reps;
  e->launches += (uint64_t)reps + 1;
  return SAME_OK;
}

int same_engine_last_timing(same_engine* e, float* h2d_ms, float* kernel_ms) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (e->in_flight) { int rc = same_engine_sync(e); if (rc) return rc; }
  if (h2d_ms) { *h2d_ms = 0.0f; if (e->timed_h2d) CK(e, cudaEventElapsedTime(h2d_ms, e->t_h2d0, e->t_h2d1)); }
  if (kernel_ms) { *kernel_ms = 0.0f; if (e->timed_kernel) CK(e, cudaEventElapsedTime(kernel_ms, e->t_k0, e->t_k1)); }
  return SAME_OK;
}

int same_engine_timer_start(same_engine* e) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  CK(e, cudaSetDevice(e->device));
  // everything submitted later starts on the copy stream (offsets/lengths/samples), so the stopwatch starts there,
  // after all earlier compute work
  CK(e, cudaEventRecord(e->t_sw1, e->compute));
  CK(e, cudaStreamWaitEvent(e->copy, e->t_sw1, 0));
  CK(e, cudaEventRecord(e->t_sw0, e->copy));
  return SAME_OK;
}

int same_engine_timer_stop(same_engine* e, float* elapsed_ms) {
  if (!e || !elapsed_ms) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  CK(e, cudaSetDevice(e->device));
  CK(e, cudaStreamSynchronize(e->copy));
  CK(e, cudaEventRecord(e->t_sw1, e->compute));
  CK(e, cudaEventSynchronize(e->t_sw1));
  CK(e, cudaEventElapsedTime(elapsed_ms, e->t_sw0, e->t_sw1));
  return SAME_OK;
}

int same_engine_get_derived(const same_engine* e, same_derived* d, float* mark_re_im, float* space_re_im, size_t cap_taps) {
  if (!e || !d) return SAME_ERR_INVALID_ARG;
  *d = e->derived;
  for (size_t i = 0; i < e->p.ntaps && i < cap_taps; ++i) {
    const float4 t = e->taps_wide.t[i];
    if (mark_re_im) { mark_re_im[2 * i] = t.x; mark_re_im[2 * i + 1] = t.y; }
    if (space_re_im) { space_re_im[2 * i] = t.z; space_re_im[2 * i + 1] = t.w; }
  }
  return SAME_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Portable stream state (format in include/same_engine.h and same_state.cu): the parts that need the engine's buffers.
// same_multi.cu reuses these helpers (same_state_* below, C++ linkage, not part of the C ABI).
// ---------------------------------------------------------------------------------------------------------------------
namespace {

// the header of a state this engine exports, and that a state it imports must match
same_state::Header state_header(const same_engine* e, uint32_t n) {
  return same_state::make_header(e->cfg, e->derived, e->taps_wide, e->p.ntaps, e->p.layout.n_words, n);
}

bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// ids -> (device id list, or nullptr + first for a contiguous run)
int upload_ids(same_engine* e, const uint32_t* ids, uint32_t n, const uint32_t** d_ids, uint32_t* first) {
  *d_ids = nullptr; *first = 0;
  if (!ids || n == 0) return SAME_OK;
  bool run = true;
  for (uint32_t i = 1; i < n && run; ++i) run = ids[i] == ids[0] + i;
  if (run) { *first = ids[0]; return SAME_OK; }
  CK(e, cudaMemcpyAsync(e->d_xids, ids, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
  *d_ids = e->d_xids;
  return SAME_OK;
}

// device -> host (pinned: one copy; pageable: through the pinned staging area)
int copy_out(same_engine* e, uint8_t* dst, const uint8_t* src, size_t bytes) {
  if (is_pinned(dst)) {
    if (bytes) CK(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, e->compute));
    return SAME_OK;
  }
  return stage_out(e, src, bytes, [&dst](const uint8_t* h, size_t n) { memcpy(dst, h, n); dst += n; });
}

// host -> device, the same way round
int copy_in(same_engine* e, uint8_t* dst, const uint8_t* src, size_t bytes) {
  if (is_pinned(src)) {
    if (bytes) CK(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, e->compute));
    return SAME_OK;
  }
  const size_t half = STAGE_BYTES / 2;
  int slot = 0;
  for (size_t off = 0; off < bytes; off += half, slot ^= 1) {
    const size_t n = std::min(half, bytes - off);
    CK(e, cudaEventSynchronize(e->stage_done[slot]));   // the copy that last read this half has finished
    memcpy(e->h_stage + slot * half, src + off, n);
    CK(e, cudaMemcpyAsync(dst + off, e->h_stage + slot * half, n, cudaMemcpyHostToDevice, e->compute));
    CK(e, cudaEventRecord(e->stage_done[slot], e->compute));
  }
  return SAME_OK;
}

int check_ids(same_engine* e, const uint32_t* ids, uint32_t n, uint32_t limit, bool unique) {
  if (!ids) return SAME_OK;
  std::vector<char> seen(unique ? limit : 0, 0);
  for (uint32_t i = 0; i < n; ++i) {
    if (ids[i] >= limit) return fail(e, SAME_ERR_INVALID_ARG, "stream id " + std::to_string(ids[i]) + " out of range");
    if (unique) {
      if (seen[ids[i]]) return fail(e, SAME_ERR_INVALID_ARG, "duplicate target stream id " + std::to_string(ids[i]));
      seen[ids[i]] = 1;
    }
  }
  return SAME_OK;
}

}  // namespace

// ---- helpers shared with same_multi.cu (the engine must be synced and the arguments checked) ----
size_t same_state_engine_record_bytes(const same_engine* e) { return same_state_record_bytes(e->p.layout.n_words); }
size_t same_state_engine_header_bytes(const same_engine* e) { return same_state::header_bytes(e->p.ntaps); }

void same_state_write_header(const same_engine* e, uint32_t n, void* dst) {
  same_state::write_header(state_header(e, n), static_cast<uint8_t*>(dst));
}

int same_state_check_header(same_engine* e, const void* buf, size_t len, uint32_t* n_records) {
  same_state::Header s;
  std::string why;
  int rc = same_state::parse_header(buf, len, &s, &why);
  if (rc == SAME_OK) rc = same_state::compare_header(state_header(e, 0), s, &why);
  if (rc != SAME_OK) return fail(e, rc, why);
  *n_records = s.n_records;
  return SAME_OK;
}

// n records of `ids` (nullptr: streams 0..n-1) -> host dst (n * record bytes); source ids are written as id + id_base
int same_state_export_records(same_engine* e, const uint32_t* ids, uint32_t n, uint32_t id_base, void* dst) {
  int rc = same_engine_sync(e);
  if (rc) return rc;
  CK(e, cudaSetDevice(e->device));
  const size_t bytes = (size_t)n * same_state_engine_record_bytes(e);
  CK(e, e->d_xfer.grow(bytes));
  CK(e, e->d_xids.grow(n));
  const uint32_t* d_ids; uint32_t first;
  rc = upload_ids(e, ids, n, &d_ids, &first);
  if (rc) return rc;
  CK(e, cudaEventRecord(e->t_st[0], e->compute));
  CK(e, same_state_launch_gather(&e->p, d_ids, first, n, id_base, e->saw_f32 ? 1u : 0u, e->d_xfer, e->compute));
  e->launches += n ? 1 : 0;
  CK(e, cudaEventRecord(e->t_st[1], e->compute));
  rc = copy_out(e, static_cast<uint8_t*>(dst), e->d_xfer, bytes);
  if (rc) return rc;
  CK(e, cudaEventRecord(e->t_st[2], e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  CK(e, cudaEventElapsedTime(&e->st_kernel_ms, e->t_st[0], e->t_st[1]));
  CK(e, cudaEventElapsedTime(&e->st_copy_ms, e->t_st[1], e->t_st[2]));
  return SAME_OK;
}

// phase 1 of an import: records -> device staging, validated there.  Changes no stream.
int same_state_import_stage(same_engine* e, uint32_t n, const void* recs, uint32_t* rec_flags) {
  int rc = same_engine_sync(e);
  if (rc) return rc;
  CK(e, cudaSetDevice(e->device));
  const size_t bytes = (size_t)n * same_state_engine_record_bytes(e);
  CK(e, e->d_xfer.grow(bytes));
  CK(e, e->d_xids.grow(n));   // for the commit, which then allocates nothing
  CK(e, e->d_xres.grow(2));
  const unsigned long long init[2] = {~0ull, 0ull};
  CK(e, cudaMemcpyAsync(e->d_xres, init, sizeof init, cudaMemcpyHostToDevice, e->compute));
  CK(e, cudaEventRecord(e->t_st[0], e->compute));
  rc = copy_in(e, e->d_xfer, static_cast<const uint8_t*>(recs), bytes);
  if (rc) return rc;
  CK(e, cudaEventRecord(e->t_st[1], e->compute));
  CK(e, same_state_launch_validate(e->d_xfer, n, e->p.layout.n_words, e->d_xres, e->compute));
  e->launches += n ? 1 : 0;
  CK(e, cudaEventRecord(e->t_st[2], e->compute));
  unsigned long long res[2];
  CK(e, cudaMemcpyAsync(res, e->d_xres, sizeof res, cudaMemcpyDeviceToHost, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  CK(e, cudaEventElapsedTime(&e->st_copy_ms, e->t_st[0], e->t_st[1]));
  CK(e, cudaEventElapsedTime(&e->st_kernel_ms, e->t_st[1], e->t_st[2]));
  if (res[0] != ~0ull) {
    const uint32_t code = (uint32_t)res[0], rec = (uint32_t)(res[0] >> 32);
    return fail(e, SAME_ERR_INVALID_ARG, "state record " + std::to_string(rec) + ": " + same_state::check_name(code));
  }
  *rec_flags = (uint32_t)res[1];
  return SAME_OK;
}

// phase 2: the staged records -> streams ids[i] (nullptr: 0..n-1); == reset(ids) + the records' state
int same_state_import_commit(same_engine* e, const uint32_t* ids, uint32_t n, uint32_t rec_flags) {
  CK(e, cudaSetDevice(e->device));
  const uint32_t* d_ids; uint32_t first;
  int rc = upload_ids(e, ids, n, &d_ids, &first);
  if (rc) return rc;
  CK(e, cudaEventRecord(e->t_st[0], e->compute));
  CK(e, same_state_launch_scatter(&e->p, d_ids, first, n, e->d_xfer, e->compute));
  e->launches += n ? 1 : 0;
  CK(e, cudaEventRecord(e->t_st[1], e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  float ms = 0.0f;
  CK(e, cudaEventElapsedTime(&ms, e->t_st[0], e->t_st[1]));
  e->st_kernel_ms += ms;
  forget_events(e, ids, n);   // they belong to the state that was replaced
  if (rec_flags & 1u) e->saw_f32 = true;
  return SAME_OK;
}

extern "C" {

size_t same_engine_state_bytes(const same_engine* e, uint32_t n) {
  return e ? same_state_engine_header_bytes(e) + (size_t)n * same_state_engine_record_bytes(e) : 0;
}

int same_engine_export_streams(same_engine* e, const uint32_t* ids, uint32_t n, void* buf, size_t cap, size_t* written) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (!ids) n = e->n_streams;
  int rc = check_ids(e, ids, n, e->n_streams, false);
  if (rc) return rc;
  const size_t need = same_engine_state_bytes(e, n);
  if (written) *written = need;
  if (!buf || cap < need) return fail(e, SAME_ERR_INVALID_ARG, "export buffer too small: " + std::to_string(need) + " bytes needed");
  same_state_write_header(e, n, buf);
  return same_state_export_records(e, ids, n, 0, static_cast<uint8_t*>(buf) + same_state_engine_header_bytes(e));
}

int same_engine_import_streams(same_engine* e, const uint32_t* ids, uint32_t n, const void* buf, size_t len) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  uint32_t n_records = 0;
  int rc = same_state_check_header(e, buf, len, &n_records);
  if (rc) return rc;
  if (!ids && n != e->n_streams) return fail(e, SAME_ERR_INVALID_ARG, "ids == NULL imports into every stream: n must equal the number of streams");
  if (n != n_records) return fail(e, SAME_ERR_INVALID_ARG, "n = " + std::to_string(n) + " but the buffer holds " + std::to_string(n_records) + " records");
  rc = check_ids(e, ids, n, e->n_streams, true);
  if (rc) return rc;
  uint32_t flags = 0;
  rc = same_state_import_stage(e, n, static_cast<const uint8_t*>(buf) + same_state_engine_header_bytes(e), &flags);
  if (rc) return rc;
  return same_state_import_commit(e, ids, n, flags);
}

int same_state_info(const void* buf, size_t len, same_config* cfg, uint32_t* n_records) {
  same_state::Header s;
  std::string why;
  const int rc = same_state::parse_header(buf, len, &s, &why);
  if (rc) return fail(nullptr, rc, why);
  if (cfg) *cfg = s.cfg;
  if (n_records) *n_records = s.n_records;
  return SAME_OK;
}

void* same_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {   // pinned for every device (same_multi)
    g_last_error = "cudaHostAlloc failed";
    return nullptr;
  }
  return p;
}
void same_host_free(void* p) { if (p) cudaFreeHost(p); }

int same_h2d_probe(int device, const void* host, size_t row_stride_bytes, size_t width_bytes, size_t rows, int reps,
                   float* elapsed_ms) {
  if (!host || !elapsed_ms || !width_bytes || !rows || reps < 1 || width_bytes > row_stride_bytes)
    return fail(nullptr, SAME_ERR_INVALID_ARG, "bad probe arguments");
  Stream st;
  Event a, b;
  DevBuf<uint8_t> d;
  cudaError_t err = cudaSetDevice(device);
  if (err == cudaSuccess) err = st.create();
  if (err == cudaSuccess) err = a.create();
  if (err == cudaSuccess) err = b.create();
  if (err == cudaSuccess) err = d.grow(width_bytes * rows);
  if (err == cudaSuccess) err = cudaMemcpy2DAsync(d, width_bytes, host, row_stride_bytes, width_bytes, rows, cudaMemcpyHostToDevice, st);  // warm-up
  if (err == cudaSuccess) err = cudaEventRecord(a, st);
  for (int i = 0; i < reps && err == cudaSuccess; ++i)
    err = cudaMemcpy2DAsync(d, width_bytes, host, row_stride_bytes, width_bytes, rows, cudaMemcpyHostToDevice, st);
  if (err == cudaSuccess) err = cudaEventRecord(b, st);
  if (err == cudaSuccess) err = cudaEventSynchronize(b);
  if (err == cudaSuccess) err = cudaEventElapsedTime(elapsed_ms, a, b);
  if (err != cudaSuccess) return fail(nullptr, SAME_ERR_CUDA, std::string("h2d probe: ") + cudaGetErrorString(err));
  return SAME_OK;
}

}  // extern "C"

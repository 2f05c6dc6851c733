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
#include <string>
#include <vector>

#include "same_params.h"

extern "C" cudaError_t same_launch_rx(const SameParams* p, const SameTaps* taps, const SameTaps2* taps2, int force_generic,
                                      uint32_t lanes_per_warp, const void* d_samples, int sample_fmt,
                                      const unsigned long long* d_offsets, const uint32_t* d_lengths,
                                      const SameTiles* tiles, cudaStream_t stream);
extern "C" cudaError_t same_launch_frontend(const SameParams* p, const int16_t* d_samples, const unsigned long long* d_offsets,
                                            const uint32_t* d_lengths, const SameTiles* tiles, cudaStream_t stream);
extern "C" cudaError_t same_launch_rx_tilefed(const SameParams* p, const SameTaps2* taps2, const uint32_t* d_lengths,
                                              const SameTiles* tiles, cudaStream_t stream);
extern "C" cudaError_t same_long_launch_dc(const SameParams* p, const int16_t* d_src, uint32_t len, float* d, uint32_t* dc_next,
                                           cudaStream_t stream);
extern "C" cudaError_t same_long_launch_commit_dc(const SameParams* p, const uint32_t* dc_next, cudaStream_t stream);
extern "C" cudaError_t same_long_launch_speculative(const SameParams* p, const SameTaps2* taps2, const float* d, uint32_t pos0,
                                                    uint32_t end, float* yfull, float* gspec, float* g_in, float* soft,
                                                    uint32_t* ctrl, cudaStream_t stream);
extern "C" cudaError_t same_launch_evsort(const same_event* d_events, uint32_t n, uint32_t n_streams, uint32_t* d_cnt,
                                          uint32_t* d_minseq, uint32_t* d_start, same_event* d_sorted, uint32_t* d_bad,
                                          cudaStream_t stream);
extern "C" cudaError_t same_launch_init(const SameParams* p, const uint32_t* d_ids, uint32_t n, int after_reset,
                                        cudaStream_t stream);
// same_state.cu
extern "C" uint32_t same_state_record_bytes(uint32_t n_words);
extern "C" uint32_t same_state_crc32(const void* data, size_t n);
extern "C" cudaError_t same_state_launch_gather(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                uint32_t id_base, uint32_t rec_flags, uint8_t* d_out, cudaStream_t stream);
extern "C" cudaError_t same_state_launch_validate(const uint8_t* d_in, uint32_t n, uint32_t n_words, unsigned long long* d_result,
                                                  cudaStream_t stream);
extern "C" cudaError_t same_state_launch_scatter(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                 const uint8_t* d_in, cudaStream_t stream);

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

size_t f32_as_usize(float x) {  // `as usize`: truncating, saturating, NaN -> 0
  if (!(x > 0.0f)) return 0;
  if (x >= 1.8e19f) return (size_t)-1;
  return (size_t)x;
}

struct InputBuf {
  uint8_t* d = nullptr; size_t cap = 0;          // device samples (s16 or f32), capacity in bytes
  unsigned long long* d_off = nullptr; uint32_t* d_len = nullptr;
  cudaEvent_t copied = nullptr, consumed = nullptr;
  bool used = false;
};

}  // namespace

struct same_engine {
  same_config cfg;
  int device = 0;
  uint32_t n_streams = 0;
  SameParams p;
  SameTaps taps;
  SameTaps2 taps2;
  int force_generic = 0;
  uint32_t lanes_per_warp = 32;   // streams per warp in the fast kernel (lane-sparse warps for small batches)
  int sm_count = 148;
  int kernel_auto = 0;            // fast-kernel flavour when force_generic == 0: 3 pipelined, 4 three-warp, 2 single-warp, 6 look-ahead
  SameTiles tiles{nullptr, nullptr, 0u, 32u, 1u};   // split pipeline (kernel 5): front-end output, allocated on first use
  size_t tiles_cap = 0;           // floats
  // long-stream path (same_long.cu): one stream, long chunks
  int long_stream = 1;            // option "long_stream"
  float *ls_d = nullptr, *ls_y = nullptr, *ls_g = nullptr, *ls_soft = nullptr, *ls_gin = nullptr;
  uint32_t* ls_ctrl = nullptr;    // device: {verified end, position reached, reason, -}
  uint32_t* ls_hctrl = nullptr;   // pinned mirror + scratch
  size_t ls_cap = 0;              // samples
  uint64_t ls_spec_launches = 0, ls_fallback_launches = 0;
  bool saw_f32 = false;           // an f32 submit happened since create / reset(all): DC state may be non-integer -> generic kernel
  uint64_t lost_events = 0, lost_payloads = 0;
  same_derived derived;
  cudaStream_t compute = nullptr, copy = nullptr;
  uint32_t* d_state = nullptr;
  StreamBlob* d_blobs = nullptr;
  same_event* d_events = nullptr;
  same_event* d_sorted = nullptr;        // arena events counting-sorted by (stream, seq) before read-back
  uint32_t* d_sort_ws = nullptr;         // cnt[n+1] | start[n+1] | minseq[n] | bad[1]
  bool pend_sorted = false;              // pend_events is one device-sorted batch: drain copies it as it is
  int device_sort = 1;                   // option "device_sort": 0 = always sort on the host (diagnostic)
  uint8_t* d_payload = nullptr;
  unsigned int* d_counters = nullptr;
  unsigned int* h_counters = nullptr;   // pinned
  uint8_t* h_stage = nullptr;           // pinned staging for event / payload read-back (STAGE_BYTES, used as two halves)
  cudaEvent_t stage_done[2] = {nullptr, nullptr};
  same_soft_symbol* d_trace = nullptr;
  uint32_t* d_ids = nullptr; size_t ids_cap = 0;
  InputBuf in[2];
  int cur = 0;
  bool in_flight = false;
  size_t events_cap = 0, payload_cap = 0;
  std::vector<same_event> pend_events;
  std::vector<uint8_t> pend_payload;
  cudaEvent_t t_h2d0 = nullptr, t_h2d1 = nullptr, t_k0 = nullptr, t_k1 = nullptr, t_sw0 = nullptr, t_sw1 = nullptr;
  bool timed_h2d = false, timed_kernel = false;
  // portable stream state (same_state.cu): device staging of records, ids, validation result, timing of the last call
  uint8_t* d_xfer = nullptr; size_t xfer_cap = 0;
  uint32_t* d_xids = nullptr; size_t xids_cap = 0;
  unsigned long long* d_xres = nullptr;
  cudaEvent_t t_st[3] = {nullptr, nullptr, nullptr};
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

int alloc_arenas(same_engine* e, size_t max_events, size_t max_payload) {
  if (e->d_events) cudaFree(e->d_events);
  if (e->d_sorted) cudaFree(e->d_sorted);
  if (e->d_payload) cudaFree(e->d_payload);
  e->d_events = nullptr; e->d_sorted = nullptr; e->d_payload = nullptr;
  CK(e, cudaMalloc(&e->d_events, max_events * sizeof(same_event)));
  CK(e, cudaMalloc(&e->d_sorted, max_events * sizeof(same_event)));
  if (!e->d_sort_ws) CK(e, cudaMalloc(&e->d_sort_ws, (3 * (size_t)e->n_streams + 3) * sizeof(uint32_t)));
  CK(e, cudaMalloc(&e->d_payload, max_payload));
  e->events_cap = max_events; e->payload_cap = max_payload;
  e->p.events = e->d_events; e->p.payload = e->d_payload;
  e->p.events_cap = (uint32_t)std::min<size_t>(max_events, 0xffffffffu);
  e->p.payload_cap = (uint32_t)std::min<size_t>(max_payload, 0xffffffffu);
  return SAME_OK;
}

static const size_t STAGE_BYTES = 2 * 48 * 32768;   // two halves of 32768 events (1.5 MiB each)

// Pull the events produced since the last collect from the device arenas into the host pending lists.
int collect(same_engine* e) {
  CK(e, cudaMemcpyAsync(e->h_counters, e->d_counters, 4 * sizeof(unsigned int), cudaMemcpyDeviceToHost, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  const size_t nev = e->h_counters[0], npay = e->h_counters[1];
  int rc = SAME_OK;
  if (nev > e->events_cap || e->h_counters[2] != 0) {
    // Events beyond the arena were dropped by the device; events whose payload did not fit were stored with
    // data_len 0 + SAME_EV_FLAG_PAYLOAD_LOST (same_transport.cuh:emit_event_impl), so everything handed to the caller
    // below stays self-consistent.  The stream state has advanced: what was dropped is lost, and counted.
    const uint64_t ev_lost = nev > e->events_cap ? nev - e->events_cap : 0;
    e->lost_events += ev_lost;
    e->lost_payloads += e->h_counters[2];
    char buf[256];
    snprintf(buf, sizeof buf, "event arena overflow since the last sync: %llu events dropped (capacity %zu), %u payloads dropped "
             "(capacity %zu bytes)", (unsigned long long)ev_lost, e->events_cap, e->h_counters[2], e->payload_cap);
    rc = fail(e, SAME_ERR_EVENT_OVERFLOW, buf);
  }
  const size_t cev = std::min(nev, e->events_cap), cpay = std::min(npay, e->payload_cap);
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
    // device -> pinned staging (two halves, so the copy of one slice overlaps the append of the other) -> pending lists
    const size_t base_ev = e->pend_events.size(), base_pay = e->pend_payload.size();
    e->pend_events.reserve(base_ev + cev);
    e->pend_payload.reserve(base_pay + cpay);
    const size_t half = STAGE_BYTES / 2;
    const uint8_t* src[2] = {reinterpret_cast<const uint8_t*>(ev_src), e->d_payload};
    const size_t bytes[2] = {cev * sizeof(same_event), cpay};
    for (int part = 0; part < 2; ++part) {
      size_t done = 0, queued = 0, qn[2] = {0, 0};
      int qslot = 0, pslot = 0, inflight = 0;
      while (done < bytes[part]) {
        while (inflight < 2 && queued < bytes[part]) {   // keep both halves in flight
          const size_t n = std::min(half, bytes[part] - queued);
          CK(e, cudaMemcpyAsync(e->h_stage + qslot * half, src[part] + queued, n, cudaMemcpyDeviceToHost, e->compute));
          CK(e, cudaEventRecord(e->stage_done[qslot], e->compute));
          qn[qslot] = n; queued += n; qslot ^= 1; ++inflight;
        }
        CK(e, cudaEventSynchronize(e->stage_done[pslot]));
        const uint8_t* h = e->h_stage + pslot * half;
        if (part == 0) {
          const same_event* ev = reinterpret_cast<const same_event*>(h);
          e->pend_events.insert(e->pend_events.end(), ev, ev + qn[pslot] / sizeof(same_event));
        } else {
          e->pend_payload.insert(e->pend_payload.end(), h, h + qn[pslot]);
        }
        done += qn[pslot]; pslot ^= 1; --inflight;
      }
    }
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

int ensure_input(same_engine* e, InputBuf& b, size_t bytes) {
  if (bytes > b.cap) {
    if (b.d) CK(e, cudaFree(b.d));
    b.d = nullptr; b.cap = 0;
    size_t cap = bytes + bytes / 8 + 8192;
    CK(e, cudaMalloc(&b.d, cap));
    b.cap = cap;
  }
  return SAME_OK;
}

// Tile buffer of the split pipeline: n_pad streams x n_max samples of f32 (+ the 34-word DC state per stream).
int ensure_tiles(same_engine* e, uint32_t max_len) {
  const uint32_t n_max = (max_len + 31u) & ~31u;
  const size_t need = (size_t)e->p.layout.n_pad * n_max;
  if (need > e->tiles_cap) {
    if (e->tiles.d) CK(e, cudaFree(e->tiles.d));
    e->tiles.d = nullptr; e->tiles_cap = 0;
    CK(e, cudaMalloc(&e->tiles.d, need * sizeof(float)));
    e->tiles_cap = need;
  }
  if (!e->tiles.dc_next) CK(e, cudaMalloc(&e->tiles.dc_next, (size_t)34 * e->p.layout.n_pad * sizeof(uint32_t)));
  e->tiles.n_max = n_max;
  return SAME_OK;
}

// ---- long-stream path: see same_long.cu ----
constexpr uint32_t kLongMinSamples = 65536;     // shorter chunks take the ordinary kernels
constexpr uint32_t kLongChunk = 1u << 24;       // samples per internal pass (bounds the scratch buffers: 16 B per sample)
constexpr uint32_t kLongSpan = 8192;            // samples per fallback launch while the AGC is locked (inside a burst)

int ensure_long(same_engine* e, size_t n) {
  if (n > e->ls_cap) {
    for (float** q : {&e->ls_d, &e->ls_y, &e->ls_g, &e->ls_soft, &e->ls_gin}) { if (*q) CK(e, cudaFree(*q)); *q = nullptr; }
    e->ls_cap = 0;
    CK(e, cudaMalloc(&e->ls_d, (n + 64) * sizeof(float)));
    CK(e, cudaMalloc(&e->ls_y, (n + 128) * sizeof(float)));
    CK(e, cudaMalloc(&e->ls_g, (n + 64) * sizeof(float)));
    CK(e, cudaMalloc(&e->ls_soft, (n + 2 * 4096 + 64) * sizeof(float)));   // + two tiles: the sequential kernel stages ahead
    CK(e, cudaMalloc(&e->ls_gin, (n / 2048 + 8) * sizeof(float)));
    e->ls_cap = n;
  }
  if (!e->ls_ctrl) CK(e, cudaMalloc(&e->ls_ctrl, 4 * sizeof(uint32_t)));
  if (!e->ls_hctrl) CK(e, cudaHostAlloc(&e->ls_hctrl, 8 * sizeof(uint32_t), cudaHostAllocDefault));
  if (!e->tiles.dc_next) CK(e, cudaMalloc(&e->tiles.dc_next, (size_t)34 * e->p.layout.n_pad * sizeof(uint32_t)));
  return SAME_OK;
}

// One stream, `len` device-resident s16 samples, on the compute stream.  Blocks the host (it steers the passes).
int run_long(same_engine* e, const int16_t* d_src, uint32_t len) {
  const SameLayout& L = e->p.layout;
  for (uint32_t base = 0; base < len; base += kLongChunk) {
    const uint32_t n = std::min(kLongChunk, len - base);
    int rc = ensure_long(e, n);
    if (rc) return rc;
    CK(e, same_long_launch_dc(&e->p, d_src + base, n, e->ls_d, e->tiles.dc_next, e->compute));
    e->launches += 1;
    uint32_t pos = 0;
    while (pos < n) {
      // is the AGC locked (inside a burst)?  then the samples are the ordinary kernel's, span by span
      CK(e, cudaMemcpyAsync(e->ls_hctrl + 4, e->d_state + (size_t)F_FLAGS * L.n_pad, sizeof(uint32_t), cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaStreamSynchronize(e->compute));
      if (e->ls_hctrl[4] & FLAG_AGC_LOCKED) {
        const uint32_t span = std::min(kLongSpan, n - pos);
        e->ls_hctrl[5] = span;
        CK(e, cudaMemcpyAsync(e->ls_ctrl + 3, e->ls_hctrl + 5, sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
        SameTiles t{e->ls_d + pos, e->tiles.dc_next, span, 1u, 0u};
        CK(e, same_launch_rx_tilefed(&e->p, &e->taps2, e->ls_ctrl + 3, &t, e->compute));
        e->launches += 1; e->ls_fallback_launches += 1;
        pos += span;
        continue;
      }
      CK(e, same_long_launch_speculative(&e->p, &e->taps2, e->ls_d, pos, n, e->ls_y, e->ls_g, e->ls_gin, e->ls_soft, e->ls_ctrl,
                                         e->compute));
      e->launches += 4; e->ls_spec_launches += 1;
      CK(e, cudaMemcpyAsync(e->ls_hctrl, e->ls_ctrl, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaStreamSynchronize(e->compute));
      const uint32_t reached = e->ls_hctrl[1];
      if (reached < pos || reached > n) return fail(e, SAME_ERR_CUDA, "long-stream pass reported an impossible position");
      if (reached == pos && e->ls_hctrl[2] == 0u) return fail(e, SAME_ERR_CUDA, "long-stream pass made no progress");
      pos = reached;
    }
    CK(e, same_long_launch_commit_dc(&e->p, e->tiles.dc_next, e->compute));
    e->launches += 1;
  }
  return SAME_OK;
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
    int rc = ensure_input(e, b, total * ssz);
    if (rc) return rc;
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
  // f32 input (now or earlier: the DC-blocker state may hold non-integers) needs the literal f32 recursion
  int kernel = e->saw_f32 ? 1 : (e->force_generic ? e->force_generic : e->kernel_auto);
  // one stream, a long chunk: the long-stream path (time-parallel DC / AGC / matched filters, sequential timing loop)
  if (e->long_stream && e->n_streams == 1 && !zeros && d_src && sample_fmt == 0 && !e->saw_f32 && e->force_generic == 0 &&
      e->p.ntaps == 42 && e->p.dc_len == 16 && lengths[0] >= kLongMinSamples) {
    int rc = run_long(e, static_cast<const int16_t*>(d_src) + offsets[0], lengths[0]);
    if (rc) return rc;
    CK(e, cudaEventRecord(e->t_k1, e->compute));
    CK(e, cudaEventRecord(b.consumed, e->compute));
    b.used = true;
    e->timed_kernel = true;
    e->in_flight = true;
    return SAME_OK;
  }
  if (kernel == 5) {
    // split pipeline: the front end needs real samples (a zeros submit has none: the fused single-warp kernel takes it,
    // the resident state is the same) and a tile buffer for the longest chunk
    if (zeros || !d_src) kernel = 2;
    else {
      uint32_t max_len = 0;
      for (uint32_t i = 0; i < e->n_streams; ++i) max_len = std::max(max_len, lengths[i]);
      int rc = ensure_tiles(e, max_len);
      if (rc) return rc;
      e->launches += 1;   // the front-end kernel
    }
  }
  CK(e, same_launch_rx(&e->p, &e->taps, &e->taps2, kernel, e->lanes_per_warp, d_src, sample_fmt, b.d_off, b.d_len, &e->tiles,
                       e->compute));
  CK(e, cudaEventRecord(e->t_k1, e->compute));
  CK(e, cudaEventRecord(b.consumed, e->compute));
  b.used = true;
  e->timed_kernel = true;
  e->launches += 1;
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
  const float sps = rate_f / kBaudHz;                                         // waveform.rs:29-31
  const size_t dc_len = f32_as_usize(cfg.dc_blocker_len * sps);               // receiver.rs:509
  const size_t ntaps = f32_as_usize(floorf(sps));                             // waveform.rs:40
  if (dc_len == 0) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "DC blocker length is 0 samples (MovingAverage::new asserts len > 0, dcblock.rs:74)");
  if (dc_len > SAME_MAX_DC) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "DC blocker longer than the engine limit of 64 samples");
  if (ntaps == 0 || ntaps > SAME_MAX_TAPS) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "matched filter length outside 1..128 taps (input_rate 521..67186 Hz)");
  uint32_t nff = cfg.eq_enabled ? cfg.eq_nff : 1u, nfb = cfg.eq_enabled ? cfg.eq_nfb : 1u;   // disabled_equalizer() receiver.rs:585-590
  float relax = cfg.eq_enabled ? cfg.eq_relaxation : 0.0f;
  float regul = cfg.eq_enabled ? cfg.eq_regularization : 1.0e-6f;
  if (nff > SAME_MAX_EQ || nfb > SAME_MAX_EQ) return fail(nullptr, SAME_ERR_INVALID_CONFIG, "equalizer order beyond the engine limit of 16 taps per arm");

  same_engine* e = new same_engine();
  e->cfg = cfg; e->device = device; e->n_streams = n_streams;
  SameParams& p = e->p;
  memset(&p, 0, sizeof p);
  memset(&e->taps, 0, sizeof e->taps);
  p.n_streams = n_streams; p.input_rate = cfg.input_rate;
  p.dc_len = (uint32_t)dc_len;
  p.dc_inv_len = 1.0f / (float)dc_len;                                        // dcblock.rs:77
  p.dc_gate = dc_len > 1 ? 1.0f : 0.0f;                                       // dcblock.rs:48
  p.agc_bw = rclampf(cfg.agc_bandwidth * sps / rate_f, 0.0f, 1.0f);           // receiver.rs:511, agc.rs:51
  p.agc_min = cfg.agc_gain_min; p.agc_max = cfg.agc_gain_max;
  p.agc_gain0 = fminf(1.0f, cfg.agc_gain_min);                                // agc.rs:55
  p.ntaps = (uint32_t)ntaps;
  cisoid_taps(p.ntaps, kMarkHz / rate_f, e->taps.mark_re, e->taps.mark_im);   // waveform.rs:41-42
  cisoid_taps(p.ntaps, kSpaceHz / rate_f, e->taps.space_re, e->taps.space_im);
  memset(&e->taps2, 0, sizeof e->taps2);
  for (uint32_t i = 0; i < p.ntaps && i < 64; ++i) {
    e->taps2.mark[i] = make_float2(e->taps.mark_re[i], e->taps.mark_im[i]);
    e->taps2.space[i] = make_float2(e->taps.space_re[i], e->taps.space_im[i]);
  }
  p.f_one = 1.0f; p.f_negzero = -0.0f;
  {
    // Kernel / mapping policy for the 22050 Hz class (measured on B200, tables in profiles/README.md), by 32-stream
    // blocks per SM:
    //  * <= 1: four-warp pipelined kernel (producer / AGC / space filter / consumer), every warp on its own scheduler:
    //    the per-stream dependent chain is what bounds the run time, so it is cut into stages.
    //  * <= 4: three-warp kernel (producer / look-ahead AGC / consumer): fewer instructions in total, still
    //    latency-hiding across the co-resident blocks.
    //  * <= 8: single-warp fast kernel (8 resident blocks per SM: the whole batch is one wave; fewest instructions).
    //  * more: single-warp look-ahead kernel (16 resident warps per SM, no d ring): the issue-bound regime.
    //  20 s streams, ms per launch, pipelined / three-warp / single-warp / look-ahead: 4096 streams 24.0 / 24.9 / 41.6 / -;
    //  8192: 36.8 / 29.1 / 43.3 / 66; 16384: 74.6 / 40.0 / 43.9 / 70; 32768: - / - / 57.7 / 81; 49152: - / - / 109 / 83;
    //  65536: 228 / 158 / 116 / 97.
    // Option "lanes_per_warp" spreads streams over more, lane-sparse warps (diagnostic).  No environment variable is
    // read here: same_engine_set_option is the only override.
    int sms = 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
    e->sm_count = sms;
    e->lanes_per_warp = 32;
    const uint32_t blocks32 = (n_streams + 31u) / 32u;
    e->kernel_auto = (blocks32 <= (uint32_t)sms) ? 3 : (blocks32 <= 4u * (uint32_t)sms) ? 4 : (blocks32 <= 8u * (uint32_t)sms) ? 2 : 6;
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

#define CKC(call)                                                                            \
  do {                                                                                       \
    cudaError_t _err = (call);                                                               \
    if (_err != cudaSuccess) {                                                               \
      int rc = fail(nullptr, SAME_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_err)); \
      same_engine_destroy(e);                                                                \
      return rc;                                                                             \
    }                                                                                        \
  } while (0)
  CKC(cudaSetDevice(device));
  CKC(cudaStreamCreateWithFlags(&e->compute, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking));
  CKC(cudaMalloc(&e->d_state, (size_t)L.n_words * L.n_pad * sizeof(uint32_t)));
  CKC(cudaMalloc(&e->d_blobs, (size_t)n_streams * sizeof(StreamBlob)));
  CKC(cudaMemsetAsync(e->d_blobs, 0, (size_t)n_streams * sizeof(StreamBlob), e->compute));
  CKC(cudaMalloc(&e->d_counters, 4 * sizeof(unsigned int)));
  CKC(cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned int), e->compute));
  CKC(cudaHostAlloc(&e->h_counters, 4 * sizeof(unsigned int), cudaHostAllocDefault));
  CKC(cudaHostAlloc(&e->h_stage, STAGE_BYTES, cudaHostAllocDefault));
  for (auto& ev : e->stage_done) CKC(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto& b : e->in) {
    CKC(cudaMalloc(&b.d_off, (size_t)n_streams * sizeof(unsigned long long)));
    CKC(cudaMalloc(&b.d_len, (size_t)n_streams * sizeof(uint32_t)));
    CKC(cudaEventCreateWithFlags(&b.copied, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&b.consumed, cudaEventDisableTiming));
  }
  CKC(cudaEventCreate(&e->t_h2d0)); CKC(cudaEventCreate(&e->t_h2d1));
  CKC(cudaEventCreate(&e->t_k0)); CKC(cudaEventCreate(&e->t_k1));
  CKC(cudaEventCreate(&e->t_sw0)); CKC(cudaEventCreate(&e->t_sw1));
  for (auto& ev : e->t_st) CKC(cudaEventCreate(&ev));
  p.state32 = e->d_state; p.blobs = e->d_blobs; p.counters = e->d_counters;
  {
    size_t nev = std::max<size_t>(65536, (size_t)n_streams * 64);
    size_t npay = std::max<size_t>(4u << 20, (size_t)n_streams * 4096);
    int rc = alloc_arenas(e, nev, npay);
    if (rc) { same_engine_destroy(e); return rc; }
  }
  CKC(same_launch_init(&e->p, nullptr, n_streams, 0, e->compute));
  CKC(cudaStreamSynchronize(e->compute));
#undef CKC
  *out = e;
  return SAME_OK;
}

void same_engine_destroy(same_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->compute) cudaStreamSynchronize(e->compute);
  if (e->copy) cudaStreamSynchronize(e->copy);
  for (auto& b : e->in) {
    if (b.d) cudaFree(b.d);
    if (b.d_off) cudaFree(b.d_off);
    if (b.d_len) cudaFree(b.d_len);
    if (b.copied) cudaEventDestroy(b.copied);
    if (b.consumed) cudaEventDestroy(b.consumed);
  }
  if (e->d_state) cudaFree(e->d_state);
  if (e->d_blobs) cudaFree(e->d_blobs);
  if (e->d_events) cudaFree(e->d_events);
  if (e->d_sorted) cudaFree(e->d_sorted);
  if (e->d_sort_ws) cudaFree(e->d_sort_ws);
  if (e->d_payload) cudaFree(e->d_payload);
  if (e->d_counters) cudaFree(e->d_counters);
  if (e->h_counters) cudaFreeHost(e->h_counters);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  for (auto& ev : e->stage_done) if (ev) cudaEventDestroy(ev);
  if (e->d_trace) cudaFree(e->d_trace);
  if (e->d_ids) cudaFree(e->d_ids);
  for (float* q : {e->ls_d, e->ls_y, e->ls_g, e->ls_soft, e->ls_gin}) if (q) cudaFree(q);
  if (e->ls_ctrl) cudaFree(e->ls_ctrl);
  if (e->ls_hctrl) cudaFreeHost(e->ls_hctrl);
  if (e->tiles.d) cudaFree(e->tiles.d);
  if (e->tiles.dc_next) cudaFree(e->tiles.dc_next);
  for (cudaEvent_t ev : {e->t_h2d0, e->t_h2d1, e->t_k0, e->t_k1, e->t_sw0, e->t_sw1}) if (ev) cudaEventDestroy(ev);
  for (cudaEvent_t ev : e->t_st) if (ev) cudaEventDestroy(ev);
  if (e->d_xfer) cudaFree(e->d_xfer);
  if (e->d_xids) cudaFree(e->d_xids);
  if (e->d_xres) cudaFree(e->d_xres);
  if (e->compute) cudaStreamDestroy(e->compute);
  if (e->copy) cudaStreamDestroy(e->copy);
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
    if (n > e->ids_cap) {
      if (e->d_ids) CK(e, cudaFree(e->d_ids));
      e->d_ids = nullptr;
      CK(e, cudaMalloc(&e->d_ids, (size_t)n * sizeof(uint32_t)));
      e->ids_cap = n;
    }
    CK(e, cudaMemcpyAsync(e->d_ids, ids, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->compute));
    CK(e, same_launch_init(&e->p, e->d_ids, n, 1, e->compute));
    e->launches += 1;
    // drop queued events of the reset streams
    std::vector<char> is_reset(e->n_streams, 0);
    for (uint32_t i = 0; i < n; ++i) is_reset[ids[i]] = 1;
    e->pend_events.erase(std::remove_if(e->pend_events.begin(), e->pend_events.end(),
                                        [&](const same_event& ev) { return is_reset[ev.stream] != 0; }),
                         e->pend_events.end());
  }
  CK(e, cudaStreamSynchronize(e->compute));
  return SAME_OK;
}

struct same_snapshot {
  int device; uint32_t n_streams; size_t state_bytes, blob_bytes;
  uint32_t* d_state; StreamBlob* d_blobs;
  bool saw_f32;   // the DC-blocker state may be non-integer: restore must keep the engine on the generic kernel
};

int same_engine_snapshot(same_engine* e, same_snapshot** out) {
  if (!e || !out) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  same_snapshot* s = new same_snapshot();
  s->device = e->device; s->n_streams = e->n_streams;
  s->state_bytes = (size_t)e->p.layout.n_words * e->p.layout.n_pad * sizeof(uint32_t);
  s->blob_bytes = (size_t)e->n_streams * sizeof(StreamBlob);
  s->d_state = nullptr; s->d_blobs = nullptr;
  s->saw_f32 = e->saw_f32;
  cudaError_t err = cudaMalloc(&s->d_state, s->state_bytes);
  if (err == cudaSuccess) err = cudaMalloc(&s->d_blobs, s->blob_bytes);
  if (err == cudaSuccess) err = cudaMemcpyAsync(s->d_state, e->d_state, s->state_bytes, cudaMemcpyDeviceToDevice, e->compute);
  if (err == cudaSuccess) err = cudaMemcpyAsync(s->d_blobs, e->d_blobs, s->blob_bytes, cudaMemcpyDeviceToDevice, e->compute);
  if (err == cudaSuccess) err = cudaStreamSynchronize(e->compute);
  if (err != cudaSuccess) {
    same_snapshot_free(s);
    return fail(e, SAME_ERR_CUDA, std::string("snapshot: ") + cudaGetErrorString(err));
  }
  *out = s;
  return SAME_OK;
}

int same_engine_restore(same_engine* e, const same_snapshot* s) {
  if (!e || !s) return fail(e, SAME_ERR_INVALID_ARG, "null argument");
  if (s->device != e->device || s->n_streams != e->n_streams ||
      s->state_bytes != (size_t)e->p.layout.n_words * e->p.layout.n_pad * sizeof(uint32_t))
    return fail(e, SAME_ERR_INVALID_ARG, "snapshot belongs to a different engine shape");
  int rc = same_engine_sync(e);
  if (rc) return rc;
  CK(e, cudaMemcpyAsync(e->d_state, s->d_state, s->state_bytes, cudaMemcpyDeviceToDevice, e->compute));
  CK(e, cudaMemcpyAsync(e->d_blobs, s->d_blobs, s->blob_bytes, cudaMemcpyDeviceToDevice, e->compute));
  CK(e, cudaStreamSynchronize(e->compute));
  e->pend_events.clear(); e->pend_payload.clear();
  e->saw_f32 = s->saw_f32;
  return SAME_OK;
}

void same_snapshot_free(same_snapshot* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->d_state) cudaFree(s->d_state);
  if (s->d_blobs) cudaFree(s->d_blobs);
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
  if (e->d_trace) { CK(e, cudaFree(e->d_trace)); e->d_trace = nullptr; }
  e->p.trace = nullptr; e->p.trace_cap = 0;
  const SameLayout& L = e->p.layout;
  CK(e, cudaMemset(e->d_state + (size_t)F_TRACE_N * L.n_pad, 0, (size_t)L.n_pad * 4));
  if (cap_per_stream) {
    CK(e, cudaMalloc(&e->d_trace, (size_t)e->n_streams * cap_per_stream * sizeof(same_soft_symbol)));
    e->p.trace = e->d_trace; e->p.trace_cap = cap_per_stream;
  }
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
    e->force_generic = value;
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
  if (strcmp(key, "kernel") == 0 || strcmp(key, "force_generic") == 0) { *value = e->force_generic; return SAME_OK; }
  if (strcmp(key, "device_sort") == 0) { *value = e->device_sort; return SAME_OK; }
  if (strcmp(key, "long_stream") == 0) { *value = e->long_stream; return SAME_OK; }
  if (strcmp(key, "long_stream_passes") == 0) { *value = (int)std::min<uint64_t>(e->ls_spec_launches, 0x7fffffff); return SAME_OK; }
  if (strcmp(key, "long_stream_fallback_spans") == 0) { *value = (int)std::min<uint64_t>(e->ls_fallback_launches, 0x7fffffff); return SAME_OK; }
  if (strcmp(key, "lanes_per_warp") == 0) { *value = (int)e->lanes_per_warp; return SAME_OK; }
  if (strcmp(key, "state_kernel_us") == 0) { *value = (int)std::min(e->st_kernel_ms * 1000.0f, 2.0e9f); return SAME_OK; }
  if (strcmp(key, "state_copy_us") == 0) { *value = (int)std::min(e->st_copy_ms * 1000.0f, 2.0e9f); return SAME_OK; }
  if (strcmp(key, "kernel_selected") == 0) {
    const bool fast_geometry = e->p.ntaps == 42 && e->p.dc_len == 16;
    *value = (e->saw_f32 || !fast_geometry) ? 1 : (e->force_generic ? e->force_generic : e->kernel_auto);
    return SAME_OK;
  }
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
    if (mark_re_im) { mark_re_im[2 * i] = e->taps.mark_re[i]; mark_re_im[2 * i + 1] = e->taps.mark_im[i]; }
    if (space_re_im) { space_re_im[2 * i] = e->taps.space_re[i]; space_re_im[2 * i + 1] = e->taps.space_im[i]; }
  }
  return SAME_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Portable stream state (format in include/same_engine.h).  The header is parsed and compared with an engine here only;
// same_multi.cu reuses these helpers (same_state_* below, C++ linkage, not part of the C ABI).
// ---------------------------------------------------------------------------------------------------------------------
namespace {

constexpr uint32_t kStMagic = 0x54534D53u;   // "SMST"
constexpr uint32_t kStVersion = 1u;
constexpr uint32_t kStBom = 0x01020304u;
constexpr size_t kStHeaderBytes = 2224;
constexpr size_t kStOffConfig = 40, kStOffDerived = 116, kStOffMark = 164, kStOffSpace = 1188, kStOffCrc = 2220;
static_assert(sizeof(same_config) == 19 * 4 && sizeof(same_derived) == 12 * 4, "4-byte fields only");
static_assert(kStOffDerived == kStOffConfig + sizeof(same_config) && kStOffMark == kStOffDerived + sizeof(same_derived) &&
              kStOffSpace == kStOffMark + 8 * SAME_MAX_TAPS && kStOffCrc + 4 == kStHeaderBytes, "header layout");

void put32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }
uint32_t get32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
// a struct of 4-byte fields <-> little-endian words
void put_words(uint8_t* p, const void* src, size_t bytes) {
  for (size_t i = 0; i < bytes; i += 4) { uint32_t v; memcpy(&v, static_cast<const uint8_t*>(src) + i, 4); put32(p + i, v); }
}
void get_words(void* dst, const uint8_t* p, size_t bytes) {
  for (size_t i = 0; i < bytes; i += 4) { const uint32_t v = get32(p + i); memcpy(static_cast<uint8_t*>(dst) + i, &v, 4); }
}

const char* const kConfigFields[19] = {
    "input_rate", "dc_blocker_len", "agc_bandwidth", "agc_gain_min", "agc_gain_max", "timing_bw_unlocked",
    "timing_bw_locked", "timing_max_deviation", "squelch_power_open", "squelch_power_close", "squelch_bandwidth",
    "preamble_max_errors", "eq_enabled", "eq_nff", "eq_nfb", "eq_relaxation", "eq_regularization",
    "frame_prefix_max_errors", "frame_max_invalid_bytes"};
const char* const kDerivedFields[12] = {"sps", "agc_bw", "agc_gain0", "samples_per_ted", "period_min", "period_max",
                                        "alpha_unlocked", "beta_unlocked", "alpha_locked", "beta_locked", "dc_len", "ntaps"};
// same_state.cu: enum Check
const char* const kCheckNames[] = {
    "valid", "CRC mismatch", "record flags (only bit 0 is defined)", "F_FLAGS (undefined bits)", "framer state > 2",
    "transport state > 2", "F_CLOCK > 2^22", "F_TEDCNT not in {0, 1}", "F_SQ_BYTECLK not in -1..7", "F_SQ_HEAD >= 64",
    "F_HIST_N > 3", "burst history length > 268", "pending length > 268", "pending kind > 2", "pending error > 3",
    "pending_offset beyond the pending text", "previous-message length > 268"};

struct StateHeader {
  same_config cfg;
  same_derived derived;
  uint8_t taps[2 * 8 * SAME_MAX_TAPS];   // raw little-endian bits: mark (re, im) x 128, then space
  uint32_t n_records, n_words, record_bytes;
};

void write_header(const same_engine* e, uint32_t n, uint8_t* h) {
  memset(h, 0, kStHeaderBytes);
  put32(h + 0, kStMagic); put32(h + 4, kStVersion); put32(h + 8, kStBom); put32(h + 12, (uint32_t)kStHeaderBytes);
  put32(h + 16, n); put32(h + 20, e->p.layout.n_words); put32(h + 24, (uint32_t)sizeof(StreamBlob));
  put32(h + 28, SAME_BURST_CAP); put32(h + 32, same_state_record_bytes(e->p.layout.n_words));
  put_words(h + kStOffConfig, &e->cfg, sizeof(same_config));
  put_words(h + kStOffDerived, &e->derived, sizeof(same_derived));
  for (uint32_t i = 0; i < e->p.ntaps; ++i) {
    const float v[4] = {e->taps.mark_re[i], e->taps.mark_im[i], e->taps.space_re[i], e->taps.space_im[i]};
    put_words(h + kStOffMark + 8 * i, v, 8);
    put_words(h + kStOffSpace + 8 * i, v + 2, 8);
  }
  put32(h + kStOffCrc, same_state_crc32(h, kStOffCrc));
}

// Format checks only (no engine): SAME_ERR_INVALID_ARG on any failure
int parse_header(const void* buf, size_t len, StateHeader* out, std::string* why) {
  const uint8_t* h = static_cast<const uint8_t*>(buf);
  auto bad = [&](const std::string& m) { *why = "state buffer: " + m; return (int)SAME_ERR_INVALID_ARG; };
  if (!h) return bad("null pointer");
  if (len < 16) return bad("truncated header");
  if (get32(h) != kStMagic) return bad("bad magic");
  if (get32(h + 8) != kStBom) return bad("wrong byte order");
  if (get32(h + 4) != kStVersion) return bad("format version " + std::to_string(get32(h + 4)) + ", this library reads version " + std::to_string(kStVersion));
  if (get32(h + 12) != kStHeaderBytes) return bad("bad header size");
  if (len < kStHeaderBytes) return bad("truncated header");
  if (get32(h + kStOffCrc) != same_state_crc32(h, kStOffCrc)) return bad("header CRC mismatch");
  StateHeader s;
  s.n_records = get32(h + 16); s.n_words = get32(h + 20); s.record_bytes = get32(h + 32);
  if (get32(h + 24) != sizeof(StreamBlob) || get32(h + 28) != SAME_BURST_CAP) return bad("stream blob layout differs from this library's");
  if (s.n_words < F_NUM_SCALARS || s.n_words > (1u << 16) || s.record_bytes != same_state_record_bytes(s.n_words))
    return bad("inconsistent record size");
  const size_t need = kStHeaderBytes + (size_t)s.n_records * s.record_bytes;
  if (len < need) return bad("truncated: " + std::to_string(len) + " bytes, the header announces " + std::to_string(need));
  if (len > need) return bad("trailing bytes after the last record");
  get_words(&s.cfg, h + kStOffConfig, sizeof(same_config));
  get_words(&s.derived, h + kStOffDerived, sizeof(same_derived));
  memcpy(s.taps, h + kStOffMark, sizeof s.taps);
  *out = s;
  return SAME_OK;
}

// The state must have been produced under exactly this engine's configuration: SAME_ERR_INVALID_CONFIG names the first
// field that differs (derived values and taps are compared bit for bit: they are libm results of the exporting host)
int compare_header(const same_engine* e, const StateHeader& s, std::string* why) {
  uint32_t a[19], b[19];
  memcpy(a, &e->cfg, sizeof a); memcpy(b, &s.cfg, sizeof b);
  for (int i = 0; i < 19; ++i)
    if (a[i] != b[i]) { *why = std::string("state was produced under another configuration: ") + kConfigFields[i] + " differs"; return SAME_ERR_INVALID_CONFIG; }
  uint32_t c[12], d[12];
  memcpy(c, &e->derived, sizeof c); memcpy(d, &s.derived, sizeof d);
  for (int i = 0; i < 12; ++i)
    if (c[i] != d[i]) { *why = std::string("derived constant ") + kDerivedFields[i] + " differs from this engine's (another host's libm?)"; return SAME_ERR_INVALID_CONFIG; }
  StateHeader mine;
  {
    uint8_t h[kStHeaderBytes];
    write_header(e, 0, h);
    memcpy(mine.taps, h + kStOffMark, sizeof mine.taps);
  }
  if (memcmp(mine.taps, s.taps, 8 * SAME_MAX_TAPS) != 0) { *why = "mark filter taps differ from this engine's"; return SAME_ERR_INVALID_CONFIG; }
  if (memcmp(mine.taps + 8 * SAME_MAX_TAPS, s.taps + 8 * SAME_MAX_TAPS, 8 * SAME_MAX_TAPS) != 0) {
    *why = "space filter taps differ from this engine's"; return SAME_ERR_INVALID_CONFIG;
  }
  if (s.n_words != e->p.layout.n_words) { *why = "state words per stream differ from this engine's"; return SAME_ERR_INVALID_CONFIG; }
  return SAME_OK;
}

bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

int ensure_xfer(same_engine* e, size_t bytes, uint32_t n_ids) {
  if (bytes > e->xfer_cap) {
    if (e->d_xfer) CK(e, cudaFree(e->d_xfer));
    e->d_xfer = nullptr; e->xfer_cap = 0;
    CK(e, cudaMalloc(&e->d_xfer, bytes));
    e->xfer_cap = bytes;
  }
  if (n_ids > e->xids_cap) {
    if (e->d_xids) CK(e, cudaFree(e->d_xids));
    e->d_xids = nullptr; e->xids_cap = 0;
    CK(e, cudaMalloc(&e->d_xids, (size_t)n_ids * sizeof(uint32_t)));
    e->xids_cap = n_ids;
  }
  if (!e->d_xres) CK(e, cudaMalloc(&e->d_xres, 2 * sizeof(unsigned long long)));
  return SAME_OK;
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

// device -> host (pinned: one copy; pageable: through the pinned staging area, two pieces in flight)
int copy_out(same_engine* e, uint8_t* dst, const uint8_t* src, size_t bytes) {
  if (is_pinned(dst)) {
    if (bytes) CK(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, e->compute));
    return SAME_OK;
  }
  const size_t half = STAGE_BYTES / 2;
  size_t done = 0, queued = 0, qn[2] = {0, 0};
  int qslot = 0, pslot = 0, inflight = 0;
  while (done < bytes) {
    while (inflight < 2 && queued < bytes) {
      const size_t n = std::min(half, bytes - queued);
      CK(e, cudaMemcpyAsync(e->h_stage + qslot * half, src + queued, n, cudaMemcpyDeviceToHost, e->compute));
      CK(e, cudaEventRecord(e->stage_done[qslot], e->compute));
      qn[qslot] = n; queued += n; qslot ^= 1; ++inflight;
    }
    CK(e, cudaEventSynchronize(e->stage_done[pslot]));
    memcpy(dst + done, e->h_stage + pslot * half, qn[pslot]);
    done += qn[pslot]; pslot ^= 1; --inflight;
  }
  return SAME_OK;
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

// ---- helpers shared with same_multi.cu (C++ linkage; the engine must be synced and the arguments checked) ----
size_t same_state_header_bytes() { return kStHeaderBytes; }
size_t same_state_engine_record_bytes(const same_engine* e) { return same_state_record_bytes(e->p.layout.n_words); }
void same_state_write_header(const same_engine* e, uint32_t n, void* dst) { write_header(e, n, static_cast<uint8_t*>(dst)); }

// header format + comparison with `e`; on failure the reason is the engine's last error
int same_state_check_header(same_engine* e, const void* buf, size_t len, uint32_t* n_records) {
  StateHeader s;
  std::string why;
  int rc = parse_header(buf, len, &s, &why);
  if (rc == SAME_OK) rc = compare_header(e, s, &why);
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
  rc = ensure_xfer(e, bytes, n);
  if (rc) return rc;
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
  rc = ensure_xfer(e, bytes, n);
  if (rc) return rc;
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
    const size_t nc = sizeof kCheckNames / sizeof kCheckNames[0];
    return fail(e, SAME_ERR_INVALID_ARG, "state record " + std::to_string(rec) + ": " + (code < nc ? kCheckNames[code] : "invalid"));
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
  // undrained events of the target streams belong to the state that was replaced
  std::vector<char> hit(e->n_streams, 0);
  for (uint32_t i = 0; i < n; ++i) hit[ids ? ids[i] : i] = 1;
  e->pend_events.erase(std::remove_if(e->pend_events.begin(), e->pend_events.end(),
                                      [&](const same_event& ev) { return hit[ev.stream] != 0; }),
                       e->pend_events.end());
  if (rec_flags & 1u) e->saw_f32 = true;
  return SAME_OK;
}

extern "C" {

size_t same_engine_state_bytes(const same_engine* e, uint32_t n) {
  return e ? kStHeaderBytes + (size_t)n * same_state_engine_record_bytes(e) : 0;
}

int same_engine_export_streams(same_engine* e, const uint32_t* ids, uint32_t n, void* buf, size_t cap, size_t* written) {
  if (!e) return fail(nullptr, SAME_ERR_INVALID_ARG, "null engine");
  if (!ids) n = e->n_streams;
  int rc = check_ids(e, ids, n, e->n_streams, false);
  if (rc) return rc;
  const size_t need = same_engine_state_bytes(e, n);
  if (written) *written = need;
  if (!buf || cap < need) return fail(e, SAME_ERR_INVALID_ARG, "export buffer too small: " + std::to_string(need) + " bytes needed");
  write_header(e, n, static_cast<uint8_t*>(buf));
  return same_state_export_records(e, ids, n, 0, static_cast<uint8_t*>(buf) + kStHeaderBytes);
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
  rc = same_state_import_stage(e, n, static_cast<const uint8_t*>(buf) + kStHeaderBytes, &flags);
  if (rc) return rc;
  return same_state_import_commit(e, ids, n, flags);
}

int same_state_info(const void* buf, size_t len, same_config* cfg, uint32_t* n_records) {
  StateHeader s;
  std::string why;
  const int rc = parse_header(buf, len, &s, &why);
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
  cudaStream_t st = nullptr; cudaEvent_t a = nullptr, b = nullptr; void* d = nullptr;
  cudaError_t err = cudaSetDevice(device);
  if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  if (err == cudaSuccess) err = cudaEventCreate(&a);
  if (err == cudaSuccess) err = cudaEventCreate(&b);
  if (err == cudaSuccess) err = cudaMalloc(&d, width_bytes * rows);
  if (err == cudaSuccess) err = cudaMemcpy2DAsync(d, width_bytes, host, row_stride_bytes, width_bytes, rows, cudaMemcpyHostToDevice, st);  // warm-up
  if (err == cudaSuccess) err = cudaEventRecord(a, st);
  for (int i = 0; i < reps && err == cudaSuccess; ++i)
    err = cudaMemcpy2DAsync(d, width_bytes, host, row_stride_bytes, width_bytes, rows, cudaMemcpyHostToDevice, st);
  if (err == cudaSuccess) err = cudaEventRecord(b, st);
  if (err == cudaSuccess) err = cudaEventSynchronize(b);
  if (err == cudaSuccess) err = cudaEventElapsedTime(elapsed_ms, a, b);
  if (d) cudaFree(d);
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  if (st) cudaStreamDestroy(st);
  if (err != cudaSuccess) return fail(nullptr, SAME_ERR_CUDA, std::string("h2d probe: ") + cudaGetErrorString(err));
  return SAME_OK;
}

}  // extern "C"

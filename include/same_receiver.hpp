// same_receiver.hpp — header-only C++ host layer over the C ABI (include/same_engine.h), mirroring the reference's
// receiver interface name for name:
//
//   same::SameReceiverBuilder   crates/sameold/src/receiver/builder.rs:14-357   (new / with_* / build)
//   same::EqualizerBuilder      builder.rs:360-437
//   same::SameReceiver          crates/sameold/src/receiver.rs:71-224           (iter_events / iter_messages / flush / reset)
//   same::SameBatchReceiver     the batched entry point (process / iter_messages_batched / decode_samedec)
//   same::SameReceiverEvent     receiver/output.rs:24-27,166-180,231-261,306-318
//   same::Message               crates/sameplace/src/message.rs:62-83
//
// The reference is Rust; no Rust toolchain exists in the build image, so this C++ layer (and the Python one in
// sameold_b200/receiver.py) is what the parity tests drive.  Link with -lsame_b200.  Errors from the engine are
// thrown as same::EngineError; decode errors are event values.
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "same_engine.h"

namespace same {

struct EngineError : std::runtime_error {
  int code;
  EngineError(int c, const std::string& what) : std::runtime_error("same_engine error " + std::to_string(c) + ": " + what), code(c) {}
};

// == sameold::Message
struct Message {
  bool is_start = false;            // StartOfMessage(header) vs EndOfMessage
  std::string text;                 // as_str()
  size_t parity_error_count = 0;    // message.rs:123
  size_t voting_byte_count = 0;     // message.rs:140
  const std::string& as_str() const { return text; }
};

// == SameReceiverEvent: what() is one of the SAME_EV_* kinds
struct SameReceiverEvent {
  uint32_t stream = 0;
  uint32_t kind = 0;
  uint64_t input_sample_counter = 0;
  uint64_t symbol_count = 0;
  uint32_t err = 0;
  std::vector<uint8_t> data;        // burst bytes (LinkState::Burst) or message text
  uint16_t parity_errors = 0, voting_bytes = 0;
  uint32_t flags = 0;

  bool is_link() const { return kind < 16; }
  const std::vector<uint8_t>* burst() const { return kind == SAME_EV_LINK_BURST ? &data : nullptr; }   // output.rs:70-75
  std::optional<Message> message_ok() const {                                                           // output.rs:58-63
    if (kind == SAME_EV_TR_MSG_SOM) return Message{true, std::string(data.begin(), data.end()), parity_errors, voting_bytes};
    if (kind == SAME_EV_TR_MSG_EOM) return Message{false, "NNNN", 0, 0};
    return std::nullopt;
  }
};

inline float rust_clamp(float x, float lo, float hi) { if (x < lo) x = lo; if (x > hi) x = hi; return x; }

class EqualizerBuilder {   // builder.rs:360-437
 public:
  EqualizerBuilder& with_filter_order(size_t nff, size_t nfb) {
    nff_ = std::max<size_t>(nff, 1); nfb_ = std::min(std::max<size_t>(nfb, 1), nff_); return *this;
  }
  EqualizerBuilder& with_relaxation(float r) { relaxation_ = rust_clamp(r, 0.0f, 1.0f); return *this; }
  EqualizerBuilder& with_regularization(float r) { regularization_ = rust_clamp(r, 0.0f, 3.40282347e+38f); return *this; }
  std::pair<size_t, size_t> filter_order() const { return {nff_, nfb_}; }
  float relaxation() const { return relaxation_; }
  float regularization() const { return regularization_; }
 private:
  size_t nff_ = 6, nfb_ = 4;
  float relaxation_ = 0.05f, regularization_ = 1.0e-6f;
};

class SameBatchReceiver;
class SameReceiver;

class SameReceiverBuilder {   // builder.rs:14-357
 public:
  explicit SameReceiverBuilder(uint32_t input_rate = 22050) { same_config_default(&cfg_, input_rate); }
  static SameReceiverBuilder samedec(uint32_t input_rate = 22050) {      // crates/samedec/src/main.rs:29-37
    SameReceiverBuilder b(input_rate); same_config_samedec(&b.cfg_, input_rate); return b;
  }
  SameReceiverBuilder& with_dc_blocker_length(float len) { cfg_.dc_blocker_len = std::fmax(0.0f, len); return *this; }
  SameReceiverBuilder& with_agc_bandwidth(float bw) { cfg_.agc_bandwidth = rust_clamp(bw, 0.0f, 1.0f); return *this; }
  SameReceiverBuilder& with_agc_gain_limits(float mn, float mx) { cfg_.agc_gain_min = mn; cfg_.agc_gain_max = mx; return *this; }
  SameReceiverBuilder& with_timing_bandwidth(float unlocked, float locked) {
    cfg_.timing_bw_unlocked = rust_clamp(unlocked, 0.0f, 1.0f);
    cfg_.timing_bw_locked = rust_clamp(locked, 0.0f, cfg_.timing_bw_unlocked); return *this;
  }
  SameReceiverBuilder& with_timing_max_deviation(float d) { cfg_.timing_max_deviation = rust_clamp(d, 0.0f, 0.5f); return *this; }
  SameReceiverBuilder& with_squelch_power(float open, float close) {
    cfg_.squelch_power_open = rust_clamp(open, 0.0f, 1.0f); cfg_.squelch_power_close = std::fmin(close, open); return *this;
  }
  SameReceiverBuilder& with_squelch_bandwidth(float bw) { cfg_.squelch_bandwidth = bw; return *this; }
  SameReceiverBuilder& with_preamble_max_errors(uint32_t e) { cfg_.preamble_max_errors = e; return *this; }
  SameReceiverBuilder& with_adaptive_equalizer(const EqualizerBuilder& eq) {
    cfg_.eq_enabled = 1; cfg_.eq_nff = (uint32_t)eq.filter_order().first; cfg_.eq_nfb = (uint32_t)eq.filter_order().second;
    cfg_.eq_relaxation = eq.relaxation(); cfg_.eq_regularization = eq.regularization(); return *this;
  }
  SameReceiverBuilder& without_adaptive_equalizer() { cfg_.eq_enabled = 0; return *this; }
  SameReceiverBuilder& with_frame_prefix_max_errors(uint32_t e) { cfg_.frame_prefix_max_errors = std::min<uint32_t>(e, 7); return *this; }
  SameReceiverBuilder& with_frame_max_invalid(uint32_t n) { cfg_.frame_max_invalid_bytes = n; return *this; }

  uint32_t input_rate() const { return cfg_.input_rate; }
  float dc_blocker_length() const { return cfg_.dc_blocker_len; }
  float agc_bandwidth() const { return cfg_.agc_bandwidth; }
  std::pair<float, float> agc_gain_limits() const { return {cfg_.agc_gain_min, cfg_.agc_gain_max}; }
  std::pair<float, float> timing_bandwidth() const { return {cfg_.timing_bw_unlocked, cfg_.timing_bw_locked}; }
  float timing_max_deviation() const { return cfg_.timing_max_deviation; }
  std::pair<float, float> squelch_power() const { return {cfg_.squelch_power_open, cfg_.squelch_power_close}; }
  float squelch_bandwidth() const { return cfg_.squelch_bandwidth; }
  uint32_t preamble_max_errors() const { return cfg_.preamble_max_errors; }
  uint32_t frame_prefix_max_errors() const { return cfg_.frame_prefix_max_errors; }
  uint32_t frame_max_invalid() const { return cfg_.frame_max_invalid_bytes; }
  const same_config& config() const { return cfg_; }

  inline SameReceiver build(int device = 0) const;                              // builder.rs:81-84
  inline SameBatchReceiver build_batch(uint32_t n_streams, int device = 0) const;
 private:
  same_config cfg_;
};

class SameBatchReceiver {
 public:
  SameBatchReceiver(const same_config& cfg, uint32_t n_streams, int device = 0) : n_(n_streams), device_(device) {
    int rc = same_engine_create(&cfg, device, n_streams, &e_);
    if (rc) throw EngineError(rc, same_last_error());
  }
  SameBatchReceiver(SameBatchReceiver&& o) noexcept : e_(o.e_), n_(o.n_), device_(o.device_) { o.e_ = nullptr; }
  SameBatchReceiver(const SameBatchReceiver&) = delete;
  ~SameBatchReceiver() { if (e_) same_engine_destroy(e_); }

  uint32_t n_streams() const { return n_; }
  uint32_t input_rate() const { return same_engine_input_rate(e_); }                               // receiver.rs:167
  std::vector<uint64_t> input_sample_counters() {                                                  // receiver.rs:175
    std::vector<uint64_t> out(n_); ck(same_engine_input_sample_counters(e_, out.data())); return out;
  }
  void reset() { ck(same_engine_reset(e_, nullptr, 0)); }                                          // receiver.rs:182-198
  void reset(const std::vector<uint32_t>& ids) { ck(same_engine_reset(e_, ids.data(), (uint32_t)ids.size())); }

  // == iter_events(chunk) driven to exhaustion on every stream; one (possibly empty) chunk per stream
  std::vector<std::vector<SameReceiverEvent>> process(const std::vector<std::vector<int16_t>>& chunks) {
    if (chunks.size() != n_) throw std::invalid_argument("one chunk per stream expected");
    std::vector<int16_t> flat; std::vector<uint64_t> off(n_); std::vector<uint32_t> len(n_);
    for (uint32_t i = 0; i < n_; ++i) { off[i] = flat.size(); len[i] = (uint32_t)chunks[i].size(); flat.insert(flat.end(), chunks[i].begin(), chunks[i].end()); }
    ck(same_engine_submit_s16(e_, flat.data(), flat.size(), off.data(), len.data()));
    ck(same_engine_sync(e_));
    return drain_by_stream();
  }
  // the reference's own item type: iter_events<I: IntoIterator<Item = f32>> (receiver.rs:119-130), any scale
  std::vector<std::vector<SameReceiverEvent>> process(const std::vector<std::vector<float>>& chunks) {
    if (chunks.size() != n_) throw std::invalid_argument("one chunk per stream expected");
    std::vector<float> flat; std::vector<uint64_t> off(n_); std::vector<uint32_t> len(n_);
    for (uint32_t i = 0; i < n_; ++i) { off[i] = flat.size(); len[i] = (uint32_t)chunks[i].size(); flat.insert(flat.end(), chunks[i].begin(), chunks[i].end()); }
    ck(same_engine_submit_f32(e_, flat.data(), flat.size(), off.data(), len.data()));
    ck(same_engine_sync(e_));
    return drain_by_stream();
  }
  std::vector<std::vector<SameReceiverEvent>> process_zeros(const std::vector<uint32_t>& lengths) {
    ck(same_engine_submit_zeros(e_, lengths.data())); ck(same_engine_sync(e_)); return drain_by_stream();
  }
  // == iter_messages (receiver.rs:155-161) for every stream
  std::vector<std::pair<uint32_t, Message>> iter_messages_batched(const std::vector<std::vector<int16_t>>& chunks) {
    std::vector<std::pair<uint32_t, Message>> out;
    for (auto& evs : process(chunks)) for (auto& e : evs) if (auto m = e.message_ok()) out.emplace_back(e.stream, *m);
    return out;
  }
  // samedec's end-of-input rule (crates/samedec/src/app.rs:71-74,103-119): flush() = up to 4 s of zeros, abandoned at
  // the first message, repeated until a whole 4 s of zeros yields no message.
  std::vector<std::vector<SameReceiverEvent>> flush_samedec() {
    const int64_t nflush = (int64_t)input_rate() * 4;
    std::vector<std::vector<SameReceiverEvent>> out(n_);
    auto c0 = input_sample_counters();
    std::vector<int64_t> pos(c0.begin(), c0.end()), origin = pos;
    std::vector<char> active(n_, 1);
    while (std::any_of(active.begin(), active.end(), [](char a) { return a != 0; })) {
      std::vector<uint32_t> lens(n_, 0);
      for (uint32_t s = 0; s < n_; ++s) if (active[s]) lens[s] = (uint32_t)(origin[s] + nflush - pos[s]);
      auto evs = process_zeros(lens);
      for (uint32_t s = 0; s < n_; ++s) {
        if (!active[s]) continue;
        pos[s] += lens[s];
        int64_t last_msg = -1;
        for (auto& e : evs[s]) { if (e.message_ok()) last_msg = (int64_t)e.input_sample_counter; out[s].push_back(std::move(e)); }
        if (last_msg >= 0) origin[s] = last_msg; else active[s] = 0;
      }
    }
    return out;
  }
  // what `samedec --file F` prints for each recording
  std::vector<std::vector<std::string>> decode_samedec(const std::vector<std::vector<int16_t>>& recordings) {
    auto a = process(recordings);
    auto b = flush_samedec();
    std::vector<std::vector<std::string>> out(n_);
    for (uint32_t s = 0; s < n_; ++s) {
      for (auto* v : {&a[s], &b[s]}) for (auto& e : *v) if (auto m = e.message_ok()) out[s].push_back(m->text);
    }
    return out;
  }
  same_engine* handle() { return e_; }
  int device() const { return device_; }

  // Portable stream state (format: same_engine.h): the complete receiver state of `ids` (empty: every stream, in order)
  std::vector<uint8_t> export_streams(const std::vector<uint32_t>& ids = {}) {
    const uint32_t n = ids.empty() ? n_ : (uint32_t)ids.size();
    std::vector<uint8_t> buf(same_engine_state_bytes(e_, n));
    size_t written = 0;
    ck(same_engine_export_streams(e_, ids.empty() ? nullptr : ids.data(), n, buf.data(), buf.size(), &written));
    return buf;
  }
  // record i -> stream ids[i] (empty: record i -> stream i); == reset(ids) + the recorded state, all or nothing
  void import_streams(const std::vector<uint8_t>& data, const std::vector<uint32_t>& ids = {}) {
    const uint32_t n = ids.empty() ? n_ : (uint32_t)ids.size();
    ck(same_engine_import_streams(e_, ids.empty() ? nullptr : ids.data(), n, data.data(), data.size()));
  }
  // a new engine built from the configuration embedded in `data`, holding every record of it
  static SameBatchReceiver from_state(const std::vector<uint8_t>& data, int device = 0) {
    same_config cfg;
    uint32_t n = 0;
    int rc = same_state_info(data.data(), data.size(), &cfg, &n);
    if (rc) throw EngineError(rc, same_last_error());
    SameBatchReceiver rx(cfg, n, device);
    rx.import_streams(data);
    return rx;
  }

 private:
  void ck(int rc) { if (rc) throw EngineError(rc, same_engine_last_error(e_)); }
  std::vector<std::vector<SameReceiverEvent>> drain_by_stream() {
    size_t nev = 0, npay = 0;
    ck(same_engine_pending(e_, &nev, &npay));
    std::vector<same_event> ev(nev); std::vector<uint8_t> pay(std::max<size_t>(npay, 1));
    if (nev) ck(same_engine_drain_events(e_, ev.data(), nev, &nev, pay.data(), pay.size(), &npay));
    std::vector<std::vector<SameReceiverEvent>> out(n_);
    for (auto& r : ev) {
      SameReceiverEvent e;
      e.stream = r.stream; e.kind = r.kind; e.input_sample_counter = r.input_sample_counter; e.symbol_count = r.symbol_count;
      e.err = r.err; e.parity_errors = r.parity_errors; e.voting_bytes = r.voting_bytes; e.flags = r.flags;
      const uint32_t n = r.kind == SAME_EV_LINK_BURST ? std::min<uint32_t>(r.data_len, SAME_BURST_CAP) : r.data_len;
      e.data.assign(pay.begin() + r.data_offset, pay.begin() + r.data_offset + n);
      out[r.stream].push_back(std::move(e));
    }
    return out;
  }
  same_engine* e_ = nullptr;
  uint32_t n_;
  int device_ = 0;
  friend class SameReceiver;
};

// == SameReceiver: a one-stream engine with the reference's method names
class SameReceiver {
 public:
  explicit SameReceiver(SameBatchReceiver&& b) : b_(std::move(b)) {}
  uint32_t input_rate() const { return b_.input_rate(); }
  uint64_t input_sample_counter() { return b_.input_sample_counters()[0]; }
  void reset() { b_.reset(); }
  // this receiver's complete state as a portable buffer
  std::vector<uint8_t> export_state() { return b_.export_streams(); }
  // == `SameReceiver: Clone` (receiver.rs:70): a new receiver on `device` (-1: this one's) in the same state
  SameReceiver clone(int device = -1) {
    return SameReceiver(SameBatchReceiver::from_state(export_state(), device < 0 ? b_.device() : device));
  }
  std::vector<SameReceiverEvent> iter_events(const std::vector<int16_t>& samples) {                                               // receiver.rs:119-130
    auto evs = b_.process(std::vector<std::vector<int16_t>>{samples});
    return std::move(evs[0]);
  }
  std::vector<SameReceiverEvent> iter_events(const std::vector<float>& samples) {                                                 // receiver.rs:119-130 (f32 items)
    auto evs = b_.process(std::vector<std::vector<float>>{samples});
    return std::move(evs[0]);
  }
  std::vector<Message> iter_messages(const std::vector<int16_t>& samples) {                                                        // receiver.rs:155-161
    std::vector<Message> out;
    for (auto& e : iter_events(samples)) if (auto m = e.message_ok()) out.push_back(*m);
    return out;
  }
  std::vector<Message> iter_messages(const std::vector<float>& samples) {
    std::vector<Message> out;
    for (auto& e : iter_events(samples)) if (auto m = e.message_ok()) out.push_back(*m);
    return out;
  }
  // receiver.rs:216-224: four seconds of zeros, the first Message, and the receiver stops AT the sample that produced it
  std::optional<Message> flush() {
    const uint32_t nflush = input_rate() * 4;
    same_snapshot* snap = nullptr;
    b_.ck(same_engine_snapshot(b_.e_, &snap));
    const uint64_t start = input_sample_counter();
    std::optional<Message> found; uint64_t at = 0;
    auto flushed = b_.process_zeros({nflush});
    for (auto& e : flushed[0]) if (auto m = e.message_ok()) { found = m; at = e.input_sample_counter; break; }
    if (found) {
      b_.ck(same_engine_restore(b_.e_, snap));
      (void)b_.process_zeros({(uint32_t)(at - start)});
    }
    same_snapshot_free(snap);
    return found;
  }
 private:
  SameBatchReceiver b_;
};

inline SameReceiver SameReceiverBuilder::build(int device) const { return SameReceiver(SameBatchReceiver(cfg_, 1, device)); }
inline SameBatchReceiver SameReceiverBuilder::build_batch(uint32_t n, int device) const { return SameBatchReceiver(cfg_, n, device); }

}  // namespace same

// same_internal.h — declarations shared between the library's translation units that are not part of the C ABI.
//
// Every file that defines or calls one of these functions includes this header, so a signature that drifts on one
// side is a compile error rather than a call through a mismatched C-linkage declaration.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stddef.h>

#include <string>

#include "same_owned.h"
#include "same_params.h"

// `as usize` of Rust: truncating, saturating, NaN -> 0
inline size_t same_f32_as_usize(float x) {
  if (!(x > 0.0f)) return 0;
  if (x >= 1.8e19f) return (size_t)-1;
  return (size_t)x;
}
// Samples per symbol and matched-filter taps at `input_rate`, in the reference's f32 arithmetic (waveform.rs:29-40)
inline float same_samples_per_symbol(uint32_t input_rate) { return (float)input_rate / 520.83f; }
inline size_t same_ntaps(uint32_t input_rate) { return same_f32_as_usize(floorf(same_samples_per_symbol(input_rate))); }

// Receiver kernels.  The values are those of the engine option "kernel" (include/same_engine.h); POLICY lets the
// engine choose from the batch size.  GENERIC takes any rate and s16 or f32 samples; the others are the fast kernels of
// the 22050 Hz class: SINGLE single-warp, PIPE five-warp pipelined, THREE three-warp, SPLIT front-end kernel followed by
// the single-warp kernel fed from its tiles, LOOKAHEAD look-ahead single-warp (16 resident warps per SM).
enum Kernel { POLICY = 0, GENERIC = 1, SINGLE = 2, PIPE = 3, THREE = 4, SPLIT = 5, LOOKAHEAD = 6 };

// ---- launchers: same_kernels.cu ----
// `kernel` is resolved by the engine (never POLICY) and only dispatched here; for GENERIC, sample_fmt (0 = int16,
// 1 = float32) picks the instantiation, and a geometry beyond SAME_GENERIC_TAPS / SAME_GENERIC_DC the wide kernel.
extern "C" cudaError_t same_launch_rx(const SameParams* p, const SameTaps* taps, const SameTaps2* taps2,
                                      const SameTapsWide* taps_wide, Kernel kernel, uint32_t lanes_per_warp, const void* d_samples, int sample_fmt,
                                      const unsigned long long* d_offsets, const uint32_t* d_lengths,
                                      const SameTiles* tiles, cudaStream_t stream);
// resident blocks per SM of `kernel` (never POLICY) at this geometry, from the runtime's occupancy calculator
extern "C" cudaError_t same_rx_resident_blocks(const SameParams* p, Kernel kernel, int* blocks);
extern "C" cudaError_t same_launch_frontend(const SameParams* p, const int16_t* d_samples, const unsigned long long* d_offsets,
                                            const uint32_t* d_lengths, const SameTiles* tiles, cudaStream_t stream);
extern "C" cudaError_t same_launch_rx_tilefed(const SameParams* p, const SameTaps2* taps2, const uint32_t* d_lengths,
                                              const SameTiles* tiles, cudaStream_t stream);
extern "C" cudaError_t same_launch_evsort(const same_event* d_events, uint32_t n, uint32_t n_streams, uint32_t* d_cnt,
                                          uint32_t* d_minseq, uint32_t* d_start, same_event* d_sorted, uint32_t* d_bad,
                                          cudaStream_t stream);
extern "C" cudaError_t same_launch_init(const SameParams* p, const uint32_t* d_ids, uint32_t n, int after_reset,
                                        cudaStream_t stream);

// ---- interleaved ingest: same_ingest.cu ----
// n_frames frames of `format` (enum same_sample_format), frame_pitch_bytes apart, columns 0..n_cols-1 from `src` on:
// column c -> row d_row[c] of `dst` (-1: none; rows dpitch samples apart, dpitch a multiple of 8), int16 rows for
// SAME_FMT_S16, f32 rows otherwise.  One launch.
extern "C" cudaError_t same_launch_ingest(uint32_t format, const void* src, uint64_t frame_pitch_bytes, uint32_t n_cols,
                                          uint32_t n_frames, const int32_t* d_row, void* dst, uint64_t dpitch,
                                          cudaStream_t stream);
// Bytes per sample of `format`, 0 for an unknown format
inline uint32_t same_format_bytes(uint32_t format) {
  return format == SAME_FMT_S16 ? 2u : format == SAME_FMT_S24 ? 3u : format == SAME_FMT_S32 || format == SAME_FMT_F32 ? 4u : 0u;
}
// The argument checks of an interleaved submit (same_engine.cu) against n_streams streams: SAME_OK, or
// SAME_ERR_INVALID_ARG with the reason (naming the channel) in *why
int same_check_interleaved(const void* frames, uint32_t format, uint32_t n_channels, uint64_t n_frames,
                           const uint32_t* channel_stream, uint32_t n_streams, std::string* why);

// ---- the long-stream path, same_long.cu: what it owns (scratch for the longest chunk so far, the control words, its
// counters) and its entry point ----
struct LongPath {
  struct Host {                  // pinned; the fields are named by the device words they travel to or from
    uint32_t verified_end, reached, why;   // <- ctrl[0..2] after a pass (same_long_seq_kernel)
    uint32_t flags;              // <- the stream's flags word (FLAG_AGC_LOCKED)
    uint32_t span;               // -> ctrl[3]: the length of an ordinary span
    unsigned long long off;      // -> off: its offset in the chunk
  };
  DevBuf<float> d, y, g, soft, g_in;   // kernels A-D: DC-blocked samples, AGC output and gains, soft symbols, block gains
  DevBuf<float> ma0, fbsum;      // general geometry: ma0 and fbsum of every sample of the chunk
  DevBuf<uint32_t> dc0;          // general geometry: the DC words the chunk started with (2 dc_len + 3)
  DevBuf<uint32_t> dc_next, dc_at;   // 22050 Hz class: A's DC-blocker state at the chunk's end, at an ordinary span's start
  DevBuf<uint32_t> ctrl;         // ctrl[0..2]: a pass's result, as in Host; ctrl + 3: the ordinary kernel's length array
  DevBuf<unsigned long long> off;   // the ordinary kernel's offset array
  PinnedBuf<Host> host;
  bool uploading = false;        // a copy from `host` is queued that no synchronisation has retired yet
  uint64_t passes = 0, fallback_spans = 0, launches = 0;   // speculative passes, ordinary spans, kernel launches
};

// One stream's `len` device-resident s16 samples through the long-stream path on `stream`, at any geometry; blocks
// the host (it steers the passes).  SAME_OK, or an error code with the message in *error.
int same_long_run(LongPath* lp, const SameParams* p, const SameTaps* taps, const SameTaps2* taps2, const SameTapsWide* taps_wide,
                  uint32_t lanes_per_warp, const int16_t* d_src, uint32_t len, cudaStream_t stream, std::string* error);

// ---- portable stream state, record format and launchers: same_state.cu ----
extern "C" uint32_t same_state_record_bytes(uint32_t n_words);
extern "C" cudaError_t same_state_launch_gather(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                uint32_t id_base, uint32_t rec_flags, uint8_t* d_out, cudaStream_t stream);
extern "C" cudaError_t same_state_launch_validate(const uint8_t* d_in, uint32_t n, uint32_t n_words, unsigned long long* d_result,
                                                  cudaStream_t stream);
extern "C" cudaError_t same_state_launch_scatter(const SameParams* p, const uint32_t* d_ids, uint32_t first, uint32_t n,
                                                 const uint8_t* d_in, cudaStream_t stream);

namespace same_state {

// Header geometry of format version 1 (include/same_engine.h), independent of the kernels' ring sizes: each filter
// section holds T = max(kMinTapSlots, ntaps) taps, the header is kFixedHeaderBytes + 16 T bytes (164 before the taps,
// 8 reserved + 4 CRC after them)
constexpr uint32_t kMinTapSlots = 128;
constexpr size_t kFixedHeaderBytes = 164 + 12;
inline constexpr uint32_t tap_slots(size_t ntaps) { return ntaps > kMinTapSlots ? (uint32_t)ntaps : kMinTapSlots; }
inline constexpr size_t header_bytes(size_t ntaps) { return kFixedHeaderBytes + 16 * (size_t)tap_slots(ntaps); }
constexpr size_t kHeaderBytes = header_bytes(0);   // 2224: every engine with at most 128 taps
static_assert(kHeaderBytes == 2224, "version-1 header of engines with at most 128 taps");

// What a state header says: the producing engine's configuration, derived constants and filter taps, and the records
// that follow
struct Header {
  same_config cfg;
  same_derived derived;
  uint32_t slots;                        // tap entries per section: tap_slots(ntaps)
  uint8_t taps[2 * 8 * SAME_MAX_TAPS];   // raw little-endian bits: mark (re, im) x slots, then space x slots
  uint32_t n_records, n_words, record_bytes;
};

Header make_header(const same_config& cfg, const same_derived& derived, const SameTapsWide& taps, uint32_t ntaps,
                   uint32_t n_words, uint32_t n_records);
void write_header(const Header& s, uint8_t* h);   // header_bytes(s.slots)
// Format checks only: SAME_ERR_INVALID_ARG on any failure, with the reason in *why
int parse_header(const void* buf, size_t len, Header* out, std::string* why);
// `theirs` must have been produced under exactly `mine`'s configuration: SAME_ERR_INVALID_CONFIG names the first field
// that differs
int compare_header(const Header& mine, const Header& theirs, std::string* why);
// text of a validate-kernel failure code
const char* check_name(uint32_t code);

}  // namespace same_state

// ---- engine-side stream-state helpers, same_engine.cu (same_multi.cu calls them; the arguments must be checked) ----
size_t same_state_engine_record_bytes(const same_engine* e);
size_t same_state_engine_header_bytes(const same_engine* e);
void same_state_write_header(const same_engine* e, uint32_t n, void* dst);
// header format + comparison with `e`; on failure the reason is the engine's last error
int same_state_check_header(same_engine* e, const void* buf, size_t len, uint32_t* n_records);
// n records of `ids` (nullptr: streams 0..n-1) -> host dst (n * record bytes); source ids are written as id + id_base
int same_state_export_records(same_engine* e, const uint32_t* ids, uint32_t n, uint32_t id_base, void* dst);
// phase 1 of an import: records -> device staging, validated there.  Changes no stream.
int same_state_import_stage(same_engine* e, uint32_t n, const void* recs, uint32_t* rec_flags);
// phase 2: the staged records -> streams ids[i] (nullptr: 0..n-1); == reset(ids) + the records' state
int same_state_import_commit(same_engine* e, const uint32_t* ids, uint32_t n, uint32_t rec_flags);

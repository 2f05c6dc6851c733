/* same_engine.h — C ABI of the B200 batched SAME receiver engine (libsame_b200.so).
 *
 * The reference (cbs228/sameold 0.6.0) is pure Rust and has NO FFI today; its public surface for this path is
 *   SameReceiverBuilder::new / with_* / build      crates/sameold/src/receiver/builder.rs:50-279
 *   SameReceiver::{iter_events, iter_messages, input_rate, input_sample_counter, reset, flush}
 *                                                   crates/sameold/src/receiver.rs:119-224
 *   SameReceiverEvent / LinkState / TransportState  crates/sameold/src/receiver/output.rs:24-27,166-180,231-261,306-318
 * Every entry point below names the reference item it replaces.  INTEGRATION.md shows the Rust `extern "C"` block and
 * the build.rs a maintainer would add so that SameReceiver (and a new iter_messages_batched) binds to this library.
 *
 * One engine = one CUDA device, one CUDA stream, N independent receivers ("streams") whose complete state
 * (receiver.rs:71-90) stays resident in HBM between submits, so chunked input == one long input, bit for bit.
 * An engine is used from one host thread at a time.  Engines on different devices share nothing.
 *
 * There is no CPU fallback: if no CUDA device is usable, same_engine_create fails with SAME_ERR_NO_DEVICE.
 */
#ifndef SAME_ENGINE_H
#define SAME_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAME_ABI_VERSION 2u

/* Status codes (the reference is infallible on this path — receiver.rs:434-436 `expect`, codesquelch.rs:230 asserts —
 * so every error here is an engine/resource error, never a decode error; decode errors are event values). */
enum same_status {
  SAME_OK = 0,
  SAME_ERR_INVALID_ARG = 1,    /* NULL pointer, stream id out of range, length too large */
  SAME_ERR_INVALID_CONFIG = 2, /* a configuration the reference would panic on (e.g. DC length 0) or beyond engine limits:
                                  matched filters of 1..512 taps (input_rate 521..267 185 Hz), DC blocker up to 512
                                  samples, equalizer up to 16 taps per arm; the message names the limit */
  SAME_ERR_NO_DEVICE = 3,      /* no usable CUDA device / device index out of range */
  SAME_ERR_CUDA = 4,           /* CUDA runtime error; see same_engine_last_error */
  SAME_ERR_EVENT_OVERFLOW = 5, /* event or payload arena too small for what was produced between two syncs: the events
                                  that fitted are still drainable and self-consistent, the rest are lost (counted by
                                  same_engine_lost_events); raise same_engine_set_event_capacity or sync more often */
  SAME_ERR_BUSY = 6            /* call not allowed while a submit is in flight (sync first) */
};

/* Mirrors SameReceiverBuilder + EqualizerBuilder field for field (builder.rs:14-29, 360-365).
 * same_config_default == SameReceiverBuilder::new(rate) (builder.rs:50-67); setters' clamping (builder.rs:95-279,
 * 393-425) is applied by same_config_sanitize and again inside same_engine_create. */
typedef struct same_config {
  uint32_t input_rate;            /* Hz                                   builder.rs:51 */
  float dc_blocker_len;           /* fraction of a symbol (0.38)          builder.rs:52,95 */
  float agc_bandwidth;            /* fraction of baud rate (0.01)         builder.rs:53,107 */
  float agc_gain_min;             /* (0.0)                                builder.rs:55,122 */
  float agc_gain_max;             /* (1.0e6)                              builder.rs:55,122 */
  float timing_bw_unlocked;       /* (0.125)                              builder.rs:56,143 */
  float timing_bw_locked;         /* (0.05)                               builder.rs:57,143 */
  float timing_max_deviation;     /* (0.01)                               builder.rs:58,162 */
  float squelch_power_open;       /* (0.10)                               builder.rs:59,190 */
  float squelch_power_close;      /* (0.05)                               builder.rs:60,190 */
  float squelch_bandwidth;        /* (0.125)                              builder.rs:61,203 */
  uint32_t preamble_max_errors;   /* (2)                                  builder.rs:62,218 */
  uint32_t eq_enabled;            /* 0 == without_adaptive_equalizer()    builder.rs:63,239 */
  uint32_t eq_nff;                /* feed-forward taps (6)                builder.rs:370,393 */
  uint32_t eq_nfb;                /* feedback taps (4)                    builder.rs:371,393 */
  float eq_relaxation;            /* NLMS mu (0.05)                       builder.rs:372,404 */
  float eq_regularization;        /* NLMS delta (1e-6)                    builder.rs:373,416 */
  uint32_t frame_prefix_max_errors; /* (2)                                builder.rs:64,256 */
  uint32_t frame_max_invalid_bytes; /* (5)                                builder.rs:65,277 */
} same_config;

/* SameReceiverBuilder::new(input_rate)  — builder.rs:50-67 */
void same_config_default(same_config* cfg, uint32_t input_rate);
/* The configuration `samedec` builds: AGC limits [1/32767, 1/200] — crates/samedec/src/main.rs:29-37 */
void same_config_samedec(same_config* cfg, uint32_t input_rate);
/* Applies the builder setters' clamping rules in place — builder.rs:95-279, 393-425 */
void same_config_sanitize(same_config* cfg);

/* Event kinds.  Link kinds == LinkState (output.rs:231-261); transport kinds == TransportState (output.rs:306-318). */
enum same_event_kind {
  SAME_EV_LINK_NOCARRIER = 0,
  SAME_EV_LINK_SEARCHING = 1,
  SAME_EV_LINK_READING = 2,
  SAME_EV_LINK_BURST = 3,        /* payload = burst bytes (LinkState::Burst(Vec<u8>)) */
  SAME_EV_TR_IDLE = 16,
  SAME_EV_TR_ASSEMBLING = 17,
  SAME_EV_TR_MSG_SOM = 18,       /* Message(Ok(StartOfMessage(hdr))): payload = header text, parity/voting counts set */
  SAME_EV_TR_MSG_EOM = 19,       /* Message(Ok(EndOfMessage)): payload = "NNNN" */
  SAME_EV_TR_MSG_ERR = 20        /* Message(Err(e)): err = 1 UnrecognizedPrefix, 2 NotAscii, 3 Malformed (sameplace message.rs:86-98) */
};

#define SAME_EV_FLAG_TRUNCATED 1u /* burst longer than the engine's burst buffer (framing.rs:152-162 has no cap);
                                     the first SAME_BURST_CAP bytes are kept — the Assembler only uses 268 (assembler.rs:169) */
#define SAME_BURST_CAP 1024u
#define SAME_EV_FLAG_PAYLOAD_LOST 2u /* the payload arena was full: the event is reported with data_len == 0 */

/* == SameReceiverEvent {what, input_sample_counter} (output.rs:24-27) plus the stream it belongs to. */
typedef struct same_event {
  uint32_t stream;               /* stream index in the engine */
  uint32_t seq;                  /* per-stream event sequence number since create/reset (order of occurrence) */
  uint64_t input_sample_counter; /* SameReceiverEvent::input_sample_counter(): samples consumed so far, 1-based */
  uint64_t symbol_count;         /* CodeAndPowerSquelch::symbol_count() when queued (codesquelch.rs:349) — diagnostic */
  uint32_t kind;                 /* enum same_event_kind */
  uint32_t err;                  /* MessageDecodeErr for SAME_EV_TR_MSG_ERR, else 0 */
  uint32_t data_offset;          /* payload position in the byte arena returned by same_engine_drain_events */
  uint32_t data_len;             /* payload bytes (true burst length even if truncated) */
  uint16_t parity_errors;        /* MessageHeader::parity_error_count (message.rs:610) */
  uint16_t voting_bytes;         /* MessageHeader::voting_byte_count  (message.rs:620) */
  uint32_t flags;                /* SAME_EV_FLAG_* */
} same_event;

/* One demodulated symbol (SymbolEstimate.data, symsync.rs:52-59) for parity checks of the soft path. */
typedef struct same_soft_symbol {
  uint64_t input_sample_counter;
  float zero;
  float sym;
} same_soft_symbol;

typedef struct same_engine same_engine;

/* == SameReceiverBuilder::build() for n_streams receivers on CUDA device `device` (receiver.rs:502-560). */
int same_engine_create(const same_config* cfg, int device, uint32_t n_streams, same_engine** out);
void same_engine_destroy(same_engine* e);
/* Library-level error text of the last failing call that had no engine (e.g. create). */
const char* same_last_error(void);
const char* same_engine_last_error(const same_engine* e);

uint32_t same_engine_num_streams(const same_engine* e);
/* == SameReceiver::input_rate (receiver.rs:167) */
uint32_t same_engine_input_rate(const same_engine* e);
/* == SameReceiver::input_sample_counter (receiver.rs:175) for each stream; `out` has n_streams entries.  Implies sync. */
int same_engine_input_sample_counters(same_engine* e, uint64_t* out);

/* == SameReceiver::reset (receiver.rs:182-198) for the listed streams (ids == NULL: all).  Implies sync. */
int same_engine_reset(same_engine* e, const uint32_t* stream_ids, uint32_t n);

/* == `SameReceiver: Clone` (receiver.rs:70): a device-resident copy of every stream's complete state.  restore puts the
 * engine back exactly where snapshot was taken (pending undrained events are dropped).  Used by the host layer to make
 * flush() stop at the sample the reference stops at (receiver.rs:220-222).  The snapshot also keeps the engine's f32 flag
 * (see same_engine_submit_f32).  Copies that leave the engine: the portable stream state below.  Both imply sync. */
typedef struct same_snapshot same_snapshot;
int same_engine_snapshot(same_engine* e, same_snapshot** out);
int same_engine_restore(same_engine* e, const same_snapshot* snap);
void same_snapshot_free(same_snapshot* snap);

/* ---- Portable stream state: `SameReceiver: Clone` (receiver.rs:70) for single streams, across engines, devices and
 * processes (checkpoint / resume, moving a stream to another slot, engine or GPU).
 *
 * An export buffer is one header followed by n records.  All fields little-endian; offsets in bytes.
 *   Header (H = 164 + 16 T + 12 bytes, T = max(128, ntaps) tap entries per filter section, ntaps =
 *   floor((f32)input_rate / 520.83f); H = 2224 up to 128 taps, 3120 at 96 kHz, 6064 at 192 kHz):
 *     0  u32 magic 0x54534D53 ("SMST")          4  u32 format version (1; readers accept only their own)
 *     8  u32 byte-order mark 0x01020304         12 u32 header size H (must match the config's input_rate)
 *     16 u32 n_records                          20 u32 n_words (state words per stream)
 *     24 u32 sizeof(StreamBlob) (3240)          28 u32 SAME_BURST_CAP
 *     32 u32 record size R                      36 u32 reserved (0)
 *     40    same_config the state was produced under (sanitized; 19 x 4 bytes)
 *     116   same_derived of that engine (12 x 4 bytes)
 *     164           mark filter taps, raw f32 bits, (re, im) x T, unused taps 0
 *     164 + 8 T     space filter taps, same layout
 *     164 + 16 T    8 bytes reserved (0)
 *     H - 4         u32 CRC-32 (zlib polynomial, as zlib.crc32) of bytes 0 .. H-5
 *   (T = 128: space taps at 1188, CRC at 2220.)
 *   Record (R = W + B bytes, W = round_up(8 + 4 * n_words, 16), B = round_up(sizeof(StreamBlob) + 4, 16)):
 *     0      u32 source stream id
 *     4      u32 flags: bit 0 = the DC-blocker state may be non-integer (the engine had an f32 submit since
 *            create / reset(all)); other bits 0
 *     8      the n_words state words in word order (independent of the engine size: a record fits any engine)
 *     W      the raw StreamBlob; zero padding in between and after
 *     R - 4  u32 CRC-32 (zlib) of record bytes 0 .. R-5
 *   At 22050 Hz (6/4 equalizer) n_words = 192 and R = 4032.
 *
 * same_engine_state_bytes: exact size of an export of n streams.
 * same_engine_export_streams: records of streams ids[0..n) in that order (ids == NULL: every stream in order, n is
 *   ignored).  Changes nothing: pending events stay pending and a stream that keeps running is bit-identical to one
 *   that was never exported.  cap too small: SAME_ERR_INVALID_ARG with *written = the size needed.  Implies sync.
 * same_engine_import_streams: record i -> stream ids[i] (ids == NULL: record i -> stream i, n == number of streams).
 *   Behaves as same_engine_reset(ids) followed by writing the records' state: undrained events of those streams are
 *   dropped, their next events continue the source's input_sample_counter and seq, their soft trace starts empty.  A
 *   record with flag bit 0 puts the engine on the rate-generic kernel until reset(all) (same results).  All or nothing:
 *   on any error no stream changes.  SAME_ERR_INVALID_ARG: bad magic, version or byte order, len not the announced
 *   size, n != n_records, an id out of range, a duplicate target id, a CRC mismatch, or a record field the receiver
 *   kernels use as an index or a length out of its range.  SAME_ERR_INVALID_CONFIG: configuration, derived constants,
 *   filter taps or words per stream differ from this engine's (the message names the first).  Implies sync.
 * same_state_info: header checks only (no engine, no GPU): the configuration and record count of a buffer. */
size_t same_engine_state_bytes(const same_engine* e, uint32_t n);
int same_engine_export_streams(same_engine* e, const uint32_t* ids, uint32_t n, void* buf, size_t cap, size_t* written);
int same_engine_import_streams(same_engine* e, const uint32_t* ids, uint32_t n, const void* buf, size_t len);
int same_state_info(const void* buf, size_t len, same_config* cfg, uint32_t* n_records);

/* Capacity of the device event arena (events) and payload arena (bytes).  The arenas fill from one same_engine_sync
 * (or any call that implies it) to the next — NOT per submit: a long run of unsynced submits accumulates.  Defaults:
 * 64 events and 4 KiB per stream, at least 65536 events / 4 MiB (a SAME stream produces ~30 events per minute).
 * On overflow sync returns SAME_ERR_EVENT_OVERFLOW once; events beyond the capacity are dropped and counted, events
 * whose payload did not fit are delivered with data_len 0 and SAME_EV_FLAG_PAYLOAD_LOST.  Implies sync. */
int same_engine_set_event_capacity(same_engine* e, size_t max_events, size_t max_payload_bytes);
/* Events dropped / payloads dropped because an arena was full, since create (cumulative). */
int same_engine_lost_events(same_engine* e, uint64_t* events_lost, uint64_t* payloads_lost);

/* Feed audio: == iter_events(input) driven to exhaustion for every stream (receiver.rs:119-130, 233-274), batched.
 * Stream i consumes samples[offsets[i] .. offsets[i]+lengths[i]) as `sa as f32` (crates/samedec/src/app.rs:112).
 * `samples` is a HOST buffer of total_samples int16 (native endian; pinned memory from same_host_alloc makes the copy
 * asynchronous); offsets/lengths have n_streams entries (length 0 = stream not fed).  Returns after enqueueing the
 * host->device copy and the kernels; the caller keeps `samples` alive until same_engine_sync returns. */
int same_engine_submit_s16(same_engine* e, const int16_t* samples, uint64_t total_samples, const uint64_t* offsets,
                           const uint32_t* lengths);
/* The natural batched layout: a HOST matrix samples[n_streams][row_stride] (int16).  Feeds columns
 * [col_start, col_start + n_cols) of every row, i.e. the same time slice of every stream, with one strided
 * host->device copy (cudaMemcpy2DAsync).  Successive calls with advancing col_start stream a long recording through the
 * engine in time-chunks; the copy of chunk k+1 overlaps the kernel of chunk k (two device buffers, two CUDA streams). */
int same_engine_submit_s16_2d(same_engine* e, const int16_t* samples, uint64_t row_stride, uint64_t col_start,
                              uint32_t n_cols);
/* Same, but `d_samples` already lives in this device's memory (no copy). */
int same_engine_submit_s16_device(same_engine* e, const int16_t* d_samples, uint64_t total_samples,
                                  const uint64_t* offsets, const uint32_t* lengths);
/* The reference's own sample type: iter_events<I: IntoIterator<Item = f32>> (receiver.rs:119-130; lib.rs:78-79 documents
 * f32 PCM at any scale — the AGC normalises).  Arbitrary f32 samples (e.g. normalised to [-1, 1]) take the literal f32
 * DC-blocker recursion (dcblock.rs:45-49,104-108) of the rate-generic kernel: the integer-exact fast path only holds
 * for integer-valued input.  After the first f32 submit an engine stays on the generic kernel until
 * same_engine_reset(all).  Host and device variants as for s16. */
int same_engine_submit_f32(same_engine* e, const float* samples, uint64_t total_samples, const uint64_t* offsets,
                           const uint32_t* lengths);
int same_engine_submit_f32_device(same_engine* e, const float* d_samples, uint64_t total_samples,
                                  const uint64_t* offsets, const uint32_t* lengths);
/* Interleaved multi-channel PCM, as audio interfaces, multi-channel WAV files and SDR channelisers deliver it:
 * `n_frames` frames of `n_channels` samples each, in one of these formats (native / little endian):
 *   SAME_FMT_S16  int16                          -> the stream gets the int16 value, exactly as same_engine_submit_s16
 *   SAME_FMT_S24  3-byte packed little-endian, sign-extended -> `sa as f32`, exact
 *   SAME_FMT_S32  int32                          -> `sa as f32`: round to nearest, ties to even (2^24 + 1 -> 2^24)
 *   SAME_FMT_F32  float                          -> the value itself
 * Sample c of frame n becomes sample n of stream channel_stream[c]: no downmix, no resampling, no scaling.
 * channel_stream == NULL maps channel c to stream c (n_channels <= n_streams); SAME_CHANNEL_SKIP drops a channel; a
 * stream no channel feeds gets no samples (as length 0 in same_engine_submit_s16).  S24, S32 and F32 channels take the
 * f32 path of same_engine_submit_f32 (the engine stays on the rate-generic kernel until same_engine_reset(all)); S16
 * channels take the s16 path, the long-stream path included.  Chunked submits equal one long submit and equal planar
 * submits of the same channels, bit for bit.
 * The frames are deinterleaved on the device: the host variant copies the bytes of the mapped channels' column range
 * [cmin, cmax] (one flat copy, or one strided cudaMemcpy2DAsync when the range is narrower than a frame) into a staging
 * buffer and converts them there, on the copy stream, overlapped with the previous submit's receiver kernel.
 * same_engine_last_timing's h2d_ms covers that copy and the conversion; the conversion counts as one launch.
 * SAME_ERR_INVALID_ARG, with nothing changed, for an unknown format, n_channels == 0, n_frames > 2^30, a stream id out
 * of range or named twice (the message names the channel), or a NULL pointer with n_frames > 0. */
enum same_sample_format { SAME_FMT_S16 = 0, SAME_FMT_S24 = 1, SAME_FMT_S32 = 2, SAME_FMT_F32 = 3 };
#define SAME_CHANNEL_SKIP 0xFFFFFFFFu
int same_engine_submit_interleaved(same_engine* e, const void* frames, uint32_t format, uint32_t n_channels,
                                   uint64_t n_frames, const uint32_t* channel_stream);
/* Same, but `d_frames` already lives in this device's memory (any alignment): no copy; the conversion runs on the
 * engine's stream (same_engine_cuda_stream), after whatever the caller queued there. */
int same_engine_submit_interleaved_device(same_engine* e, const void* d_frames, uint32_t format, uint32_t n_channels,
                                          uint64_t n_frames, const uint32_t* channel_stream);
/* Feed lengths[i] zero samples to stream i: the body of SameReceiver::flush (receiver.rs:216-224) without its early
 * return; the host layer applies samedec's repeat-until-quiet rule (app.rs:71-74,118). */
int same_engine_submit_zeros(same_engine* e, const uint32_t* lengths);
/* Wait for everything submitted; makes its events drainable. */
int same_engine_sync(same_engine* e);

/* Number of events / payload bytes waiting to be drained (after sync). */
int same_engine_pending(same_engine* e, size_t* n_events, size_t* n_payload_bytes);
/* Copies out all pending events sorted by (stream, seq) — per-stream order of occurrence, as iter_events yields them —
 * and their payload bytes; clears the pending set.  If a capacity is too small nothing is consumed and
 * SAME_ERR_INVALID_ARG is returned (query same_engine_pending first). */
int same_engine_drain_events(same_engine* e, same_event* events, size_t events_cap, size_t* n_events, uint8_t* payload,
                             size_t payload_cap, size_t* n_payload);

/* Optional soft-symbol trace (diagnostic tap; SURVEY.md §5 "tracing"): keep up to cap_per_stream symbols per stream
 * per drain.  0 disables.  Implies sync. */
int same_engine_enable_soft_trace(same_engine* e, uint32_t cap_per_stream);
int same_engine_read_soft_trace(same_engine* e, uint32_t stream, same_soft_symbol* out, size_t cap, size_t* n);

/* Engine options (diagnostic; every setting must produce identical results, the tests cross-check them).  The library
 * reads no environment variables: this call is the only way to override the measured kernel policy.
 *   "kernel"          0 engine picks the kernel from the batch size (default); 1 rate-generic kernel even where the
 *                     22050 Hz fast kernels apply; 2 single-warp fast kernel; 3 five-warp pipelined kernel;
 *                     4 three-warp kernel; 5 split pipeline: the time-parallel front-end kernel (s16 -> exact DC-blocked
 *                     f32 tiles, HBM-bound) followed by the single-warp kernel fed from those tiles -- the measured
 *                     alternative to the fused kernels (DESIGN.md section 5); 6 look-ahead single-warp kernel (throughput
 *                     regime: 16 resident warps per SM).  ("force_generic": old name.)
 *   "long_stream"     1 (default): an engine with ONE stream sends chunks of >= 65536 s16 samples down the long-stream
 *                     path (same_long.cu: DC blocker, AGC and matched filters time-parallel, timing loop sequential;
 *                     such a submit returns when the chunk is done), at any geometry the engine accepts, s16 only: not
 *                     after an f32 submit since create / reset(all), nor with option "kernel" set; 0: always the
 *                     ordinary kernels
 *   "lanes_per_warp"  streams per warp of the fast kernels (1..32)
 *   "device_sort"     1 (default): big batches of events are put into per-stream order on the device before the
 *                     read-back; 0: always on the host
 * Implies sync. */
int same_engine_set_option(same_engine* e, const char* key, int value);
/* Reads an option back; additionally "kernel_selected": the kernel the next s16 submit will launch (1 generic,
 * 2 single-warp, 3 pipelined, 4 three-warp, 6 look-ahead single-warp) — the policy result for this batch size unless
 * "kernel" overrides it; "rollbacks": how often the pipelined kernel's timing warp resumed a stream from a symbol whose
 * symbol stages changed its state (sync found or end of a burst), counted up to the last sync (diagnostic);
 * "resident_blocks_per_sm": how many blocks of that kernel (each serves 32 streams) fit on one SM at this engine's
 * geometry, from the CUDA runtime's occupancy calculator (registers, shared memory, block limits). */
int same_engine_get_option(same_engine* e, const char* key, int* value);

/* Measurement aid: runs only the front-end kernel (feed-forward stages: s16 -> f32, DC blocker; 2 B read + 4 B written
 * per sample) `reps` times on device-resident samples and returns its CUDA-event time per launch.  The resident
 * receiver state is not changed. */
int same_engine_frontend_probe(same_engine* e, const int16_t* d_samples, uint64_t total_samples, const uint64_t* offsets,
                               const uint32_t* lengths, int reps, float* ms_per_launch);
/* Timing of the last completed submit, measured with CUDA events on the engine's stream: host->device copy (for an
 * interleaved submit: the copy and the conversion to planar rows) and receiver kernel, in milliseconds; kernel launch
 * count since create (for bench.py's gpu_launches). */
int same_engine_last_timing(same_engine* e, float* h2d_ms, float* kernel_ms);
uint64_t same_engine_launch_count(const same_engine* e);
/* Device-side stopwatch over everything submitted between start and stop (host->device copies, kernels), taken with
 * CUDA events on the engine's own streams.  timer_stop waits for the work to finish (it does not drain events). */
int same_engine_timer_start(same_engine* e);
int same_engine_timer_stop(same_engine* e, float* elapsed_ms);
/* cudaStream_t of the engine (as void*), so callers can order their own device work (e.g. a generator) before submit. */
void* same_engine_cuda_stream(same_engine* e);

/* Pinned host memory for sample buffers (pinned for every device of the process). */
void* same_host_alloc(size_t bytes);
void same_host_free(void* p);
/* Measurement aid: the bare host->device copy ceiling of this process on `device` — `reps` strided copies of `rows`
 * rows of `width_bytes` (source pitch `row_stride_bytes`; width == pitch makes it one flat copy) from pinned `host`
 * into a scratch device buffer, no kernel, timed with CUDA events.  bench.py runs it on every rank at once to get the
 * box's aggregate pinned H2D rate that the end-to-end numbers are bounded by. */
int same_h2d_probe(int device, const void* host, size_t row_stride_bytes, size_t width_bytes, size_t rows, int reps,
                   float* elapsed_ms);

/* Derived constants as the engine computed them on the host (receiver.rs:502-560), for parity tests. */
typedef struct same_derived {
  float sps, agc_bw, agc_gain0, samples_per_ted, period_min, period_max;
  float alpha_unlocked, beta_unlocked, alpha_locked, beta_locked;
  uint32_t dc_len, ntaps;
} same_derived;
int same_engine_get_derived(const same_engine* e, same_derived* d, float* mark_re_im, float* space_re_im, size_t cap_taps);

uint32_t same_abi_version(void);

/* ---------------------------------------------------------------------------------------------------------------------
 * Several devices in one process (north_star: "streams shard naturally across the 8 GPUs of one box, with one host
 * thread and CUDA stream per device ... no NCCL").  same_multi owns one engine and one host thread per entry of
 * `devices` (a device may be listed more than once); shard i holds the contiguous global stream range
 * [n_streams*i/n_devices, n_streams*(i+1)/n_devices).  Every call fans out to the shards' threads and returns when all
 * of them have enqueued (submit) or finished (sync, drain).  Semantics per stream are those of the single-device calls
 * above; events come back with GLOBAL stream ids, sorted by (stream, order of occurrence).  This is what a Rust
 * iter_messages_batched over a whole box calls (bindings/rust/src/batched.rs).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct same_multi same_multi;
int same_multi_create(const same_config* cfg, const int* devices, uint32_t n_devices, uint32_t n_streams, same_multi** out);
void same_multi_destroy(same_multi* m);
const char* same_multi_last_error(const same_multi* m);
uint32_t same_multi_num_shards(const same_multi* m);
uint32_t same_multi_num_streams(const same_multi* m);
int same_multi_shard_info(const same_multi* m, uint32_t shard, int* device, uint32_t* first_stream, uint32_t* n_streams);
/* The engine of one shard, for per-device settings and timers (same_engine_set_option, same_engine_timer_*). */
same_engine* same_multi_engine(same_multi* m, uint32_t shard);
/* offsets/lengths have n_streams (global) entries; each device copies only the span of `samples` its streams touch. */
int same_multi_submit_s16(same_multi* m, const int16_t* samples, uint64_t total_samples, const uint64_t* offsets,
                          const uint32_t* lengths);
int same_multi_submit_f32(same_multi* m, const float* samples, uint64_t total_samples, const uint64_t* offsets,
                          const uint32_t* lengths);
/* HOST matrix samples[n_streams][row_stride]: device i takes its own rows, columns [col_start, col_start + n_cols). */
int same_multi_submit_s16_2d(same_multi* m, const int16_t* samples, uint64_t row_stride, uint64_t col_start,
                             uint32_t n_cols);
/* Interleaved frames (same_engine_submit_interleaved) with GLOBAL stream ids in channel_stream: each device copies and
 * converts only the column range of its own streams' channels. */
int same_multi_submit_interleaved(same_multi* m, const void* frames, uint32_t format, uint32_t n_channels,
                                  uint64_t n_frames, const uint32_t* channel_stream);
int same_multi_submit_zeros(same_multi* m, const uint32_t* lengths);
int same_multi_sync(same_multi* m);
int same_multi_reset(same_multi* m);
int same_multi_input_sample_counters(same_multi* m, uint64_t* out);
int same_multi_pending(same_multi* m, size_t* n_events, size_t* n_payload_bytes);
int same_multi_drain_events(same_multi* m, same_event* events, size_t events_cap, size_t* n_events, uint8_t* payload,
                            size_t payload_cap, size_t* n_payload);
/* Portable stream state with GLOBAL stream ids (format and semantics as same_engine_*_streams above), routed to the
 * owning shards and run on the shards' threads in parallel; records come out in the order of `ids` and carry global
 * source ids.  An import validates on every shard before any shard changes. */
size_t same_multi_state_bytes(const same_multi* m, uint32_t n);
int same_multi_export_streams(same_multi* m, const uint32_t* ids, uint32_t n, void* buf, size_t cap, size_t* written);
int same_multi_import_streams(same_multi* m, const uint32_t* ids, uint32_t n, const void* buf, size_t len);

#ifdef __cplusplus
}
#endif
#endif /* SAME_ENGINE_H */

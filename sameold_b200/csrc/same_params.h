// same_params.h — constants and per-stream state layout shared by the host engine and the device kernels.
//
// HBM data layout (DESIGN.md §3):
//   * state32: structure-of-arrays of 32-bit words, word w of stream s at state32[w * n_pad + s] (n_pad = n_streams
//     rounded up to 32) so that a warp (= 32 consecutive streams) loads/stores every field fully coalesced.
//   * blobs:   one StreamBlob per stream (array-of-structs) holding the byte-oriented, event-rate transport state
//     (burst history, pending/previous message, burst under construction).  Touched only at burst/message rate.
//   * events / payload arena: appended with atomics, drained by the host after sync.
#pragma once

#include <stdint.h>

#include <vector_types.h>

#include "../../include/same_engine.h"

#define SAME_MAX_TAPS 128      // matched filter taps (floor(rate/520.83)): 42 @22050, 84 @44100, 92 @48000
#define SAME_MAX_DC 64         // DC blocker length ((0.38*sps) as usize): 16 @22050, 32 @44100, 35 @48000
#define SAME_MAX_EQ 16         // equalizer taps per arm
#define SAME_SQ_HIST 64        // codesquelch.rs:145 sample history
#define SAME_MAX_MESSAGE_LENGTH 268  // assembler.rs:70

// Scalar fields of state32 (one word each)
enum SameField {
  F_AGC_GAIN = 0,
  F_FLAGS,        // see FLAG_* below
  F_CLOCK,        // ted_sample_clock                         receiver.rs:87
  F_UNTIL,        // samples_until_next_ted                   receiver.rs:88
  F_PAVG,         // TimingLoop::period_avg                   symsync.rs:122
  F_PINST,        // TimingLoop::period_inst                  symsync.rs:125
  F_TED0, F_TED1, F_TED2,  // ZeroCrossingTed::history        symsync.rs:250
  F_TEDCNT,       // ZeroCrossingTed::sample_counter          symsync.rs:251
  F_SQ_DATA,      // CodeCorrelator::data                     codesquelch.rs:400
  F_SQ_POWER,     // PowerTracker::power                      codesquelch.rs:456
  F_SQ_PFLAGS,    // power_history as a 32-bit shift register codesquelch.rs:148 (bit 31 newest, bit 0 oldest)
  F_SQ_BYTECLK,   // sample_clock: -1 None, else 0..7         codesquelch.rs:154
  F_SYMCOUNT_LO, F_SYMCOUNT_HI,  // symbol_counter            codesquelch.rs:151
  F_N_LO, F_N_HI, // input_sample_counter                     receiver.rs:83
  F_EQ_TRAIN_SA, F_EQ_TRAIN_CNT,  // EnabledTraining(u32,u32) equalize.rs:346
  F_FR_WORD, F_FR_COUNT, F_FR_INVALID, F_FR_MSGLEN,  // Framer State payloads  framing.rs:206-222
  F_EOM_LO, F_EOM_HI,  // force_eom_at_sample                 receiver.rs:89
  F_TRNEXT_LO, F_TRNEXT_HI,  // earliest assembler deadline (cache: min of pending and history deadlines)
  F_HIST_N,       // assembler burst history length (0..3)    assembler.rs:113
  F_SEQ,          // per-stream event sequence number
  F_TRACE_N,      // soft-trace fill
  F_DC_FFSUM, F_DC_FBSUM,  // MovingAverage::moving_sum       dcblock.rs:65
  F_SQ_HEAD,      // next write slot (== oldest entry) of the in-place squelch history ring `sqh`
  F_NUM_SCALARS
};

// F_FLAGS bits
#define FLAG_AGC_LOCKED   (1u << 0)   // agc.rs:29
#define FLAG_SQ_LOCK      (1u << 1)   // codesquelch.rs:157
#define FLAG_BW_LOCKED    (1u << 2)   // which (alpha,beta) pair the timing loop uses (symsync.rs:176-180)
#define FLAG_EQ_TRAINING  (1u << 3)   // EqualizerState::EnabledTraining vs EnabledFeedback (equalize.rs:336-347)
#define FLAG_FORCE_EOM    (1u << 4)   // force_eom_at_sample.is_some()
#define FLAG_PENDING      (1u << 5)   // PendingResult::Pending      assembler.rs:280
#define FLAG_HAVE_PREV    (1u << 6)   // Assembler::previous.is_some()
#define FLAG_FR_SHIFT     8           // 2 bits: 0 Idle, 1 PrefixSearch, 2 DataRead   framing.rs:206
#define FLAG_LINK_SHIFT   10          // 2 bits: last reported LinkState kind        receiver.rs:84
#define FLAG_TR_SHIFT     12          // 2 bits: last reported TransportState kind   receiver.rs:85 (0 Idle 1 Assembling 2 Message)

// Layout of the array fields, computed once per engine from the configuration
struct SameLayout {
  uint32_t n_pad;       // streams rounded up to a multiple of 32
  uint32_t dc_ff;       // [dc_len]  ff MovingAverage window, oldest first
  uint32_t dc_fb;       // [dc_len]
  uint32_t win;         // [ntaps]   FskDemod window, oldest first
  uint32_t sqh;         // [64]      squelch sample history, ring in place: oldest entry at slot F_SQ_HEAD
  uint32_t eq_ffc, eq_fbc, eq_ffw, eq_fbw;  // equalizer taps and windows (windows oldest first)
  uint32_t n_words;     // total words per stream
};

struct BurstSlot {              // TimedData<Burst>  assembler.rs:98, timeddata.rs:3-9
  unsigned long long deadline;
  uint32_t len;
  uint8_t data[SAME_MAX_MESSAGE_LENGTH];
};

struct StreamBlob {
  BurstSlot hist[3];                       // BurstHistory (<= 3 entries, oldest first)   assembler.rs:353
  unsigned long long pending_deadline;     // PendingResult::Pending(TimedData)           assembler.rs:280
  unsigned long long prev_deadline;        // PreviousMessage                             assembler.rs:356
  uint16_t pending_len, pending_parity, pending_voting, pending_offset;
  uint8_t pending_kind;                    // 0 SOM, 1 EOM, 2 Err
  uint8_t pending_err;
  uint16_t prev_len;
  uint32_t pad0;
  uint8_t pending_text[SAME_MAX_MESSAGE_LENGTH];
  uint8_t prev_text[SAME_MAX_MESSAGE_LENGTH];
  uint8_t est[SAME_MAX_MESSAGE_LENGTH];    // scratch of combiner::estimate_message (bytes / burst counts / bit errors)
  uint8_t est_nb[SAME_MAX_MESSAGE_LENGTH];
  uint8_t est_err[SAME_MAX_MESSAGE_LENGTH];
  uint8_t burst[SAME_BURST_CAP];           // Framer State::DataRead(Vec<u8>, _)          framing.rs:221
};

// Everything the kernels need that is uniform over streams (lives in __constant__ memory)
struct SameParams {
  SameLayout layout;
  uint32_t n_streams;
  uint32_t input_rate;
  // DC blocker                                                dcblock.rs
  uint32_t dc_len;
  float dc_inv_len;
  float dc_gate;          // (len > 1) as u8 as f32            dcblock.rs:48
  // AGC                                                       agc.rs:49-57
  float agc_bw, agc_min, agc_max, agc_gain0;
  // demod                                                     waveform.rs:39-64
  uint32_t ntaps;
  // timing loop                                               symsync.rs:142-163, 329-337
  float spt, pmin, pmax, alpha_u, beta_u, alpha_l, beta_l;
  // squelch                                                   codesquelch.rs:189-210
  uint32_t sq_sync_word, sq_max_err;
  float sq_open, sq_close, sq_bw;
  // equalizer                                                 equalize.rs:124-151, receiver.rs:524-534,585-590
  uint32_t eq_nff, eq_nfb;
  float eq_relax, eq_regul;
  // framer                                                    framing.rs:71-78
  uint32_t fr_max_prefix_err, fr_max_invalid;
  // transport                                                 assembler.rs:85,92; receiver.rs:496
  unsigned long long interburst_symbols, history_symbols, force_eom_samples;
  // output arenas
  same_event* events;
  uint8_t* payload;
  unsigned int* counters;         // [0] events appended, [1] payload bytes appended, [2] payloads dropped (arena full),
                                  // [3] roll-backs of the pipelined kernel (same_rx_pipe_kernel)
  uint32_t events_cap, payload_cap;
  same_soft_symbol* trace;        // [n_streams][trace_cap] or null
  uint32_t trace_cap;
  // per-stream state
  uint32_t* state32;
  StreamBlob* blobs;
  // 1.0f and -0.0f as RUN-TIME values: fma(a, f_one, b) and fma(a, b, f_negzero) are the exact add / exact multiply of
  // the packed FFMA2 path; as compile-time constants ptxas would fold them and re-fuse the pair (it contracts packed
  // mul+add even with --fmad=false)
  float f_one, f_negzero;
};

// Output of the front-end kernel (same_frontend_kernel), input of the tile-fed loop kernel: exact DC-blocked f32 samples
// in lane-major tiles, sample n of stream s at d[((s / 32) * n_max + n) * 32 + (s % 32)], plus the DC-blocker state the
// front end leaves behind (34 words per stream, word-major like state32).
struct SameTiles {
  float* d;
  uint32_t* dc_next;
  uint32_t n_max;      // samples per stream in the tile buffer (multiple of 32)
  uint32_t stride;     // floats between consecutive samples of one stream: 32 (lane-major tiles) or 1 (one dense stream:
                       // the long-stream path, same_long.cu)
  uint32_t commit_dc;  // the tile-fed loop kernel copies dc_next into the state words when it finishes (0: the caller
                       // does it later -- the kernel only covers a span of the front end's output)
};

struct SameTaps2 {                // the same taps as (re, im) pairs for the packed-FFMA2 matched filter
  float2 mark[64], space[64];
};

struct SameTaps {                 // matched filter taps, tap i pairs with the sample i steps back from the newest
  float mark_re[SAME_MAX_TAPS], mark_im[SAME_MAX_TAPS], space_re[SAME_MAX_TAPS], space_im[SAME_MAX_TAPS];
};

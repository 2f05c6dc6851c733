//! Raw bindings to include/same_engine.h (ABI version 2).  Field order and types match the C header exactly.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct same_config {
    pub input_rate: u32,
    pub dc_blocker_len: f32,
    pub agc_bandwidth: f32,
    pub agc_gain_min: f32,
    pub agc_gain_max: f32,
    pub timing_bw_unlocked: f32,
    pub timing_bw_locked: f32,
    pub timing_max_deviation: f32,
    pub squelch_power_open: f32,
    pub squelch_power_close: f32,
    pub squelch_bandwidth: f32,
    pub preamble_max_errors: u32,
    pub eq_enabled: u32,
    pub eq_nff: u32,
    pub eq_nfb: u32,
    pub eq_relaxation: f32,
    pub eq_regularization: f32,
    pub frame_prefix_max_errors: u32,
    pub frame_max_invalid_bytes: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct same_event {
    pub stream: u32,
    pub seq: u32,
    pub input_sample_counter: u64,
    pub symbol_count: u64,
    pub kind: u32,
    pub err: u32,
    pub data_offset: u32,
    pub data_len: u32,
    pub parity_errors: u16,
    pub voting_bytes: u16,
    pub flags: u32,
}

pub const SAME_EV_LINK_NOCARRIER: u32 = 0;
pub const SAME_EV_LINK_SEARCHING: u32 = 1;
pub const SAME_EV_LINK_READING: u32 = 2;
pub const SAME_EV_LINK_BURST: u32 = 3;
pub const SAME_EV_TR_IDLE: u32 = 16;
pub const SAME_EV_TR_ASSEMBLING: u32 = 17;
pub const SAME_EV_TR_MSG_SOM: u32 = 18;
pub const SAME_EV_TR_MSG_EOM: u32 = 19;
pub const SAME_EV_TR_MSG_ERR: u32 = 20;

#[repr(C)]
pub struct same_engine {
    _private: [u8; 0],
}

/// Opaque handle: one batch sharded over several devices (one engine + one host thread per device).
#[repr(C)]
pub struct same_multi {
    _private: [u8; 0],
}

/// Opaque copy of the resident state of all streams (`SameReceiver: Clone`, receiver.rs:70).
#[repr(C)]
pub struct same_snapshot {
    _private: [u8; 0],
}

/// One demodulated symbol (SymbolEstimate.data, symsync.rs:52-59): diagnostic tap.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct same_soft_symbol {
    pub input_sample_counter: u64,
    pub zero: f32,
    pub sym: f32,
}

/// Constants the engine derived from the configuration (for parity checks against the CPU receiver).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct same_derived {
    pub sps: f32,
    pub agc_bw: f32,
    pub agc_gain0: f32,
    pub samples_per_ted: f32,
    pub period_min: f32,
    pub period_max: f32,
    pub alpha_unlocked: f32,
    pub beta_unlocked: f32,
    pub alpha_locked: f32,
    pub beta_locked: f32,
    pub dc_len: u32,
    pub ntaps: u32,
}

extern "C" {
    pub fn same_abi_version() -> u32;
    pub fn same_config_default(cfg: *mut same_config, input_rate: u32);
    pub fn same_config_samedec(cfg: *mut same_config, input_rate: u32);
    pub fn same_config_sanitize(cfg: *mut same_config);
    pub fn same_engine_create(cfg: *const same_config, device: c_int, n_streams: u32, out: *mut *mut same_engine) -> c_int;
    pub fn same_engine_destroy(e: *mut same_engine);
    pub fn same_last_error() -> *const c_char;
    pub fn same_engine_last_error(e: *const same_engine) -> *const c_char;
    pub fn same_engine_num_streams(e: *const same_engine) -> u32;
    pub fn same_engine_input_rate(e: *const same_engine) -> u32;
    pub fn same_engine_input_sample_counters(e: *mut same_engine, out: *mut u64) -> c_int;
    pub fn same_engine_reset(e: *mut same_engine, stream_ids: *const u32, n: u32) -> c_int;
    pub fn same_engine_submit_s16(e: *mut same_engine, samples: *const i16, total_samples: u64, offsets: *const u64, lengths: *const u32) -> c_int;
    pub fn same_engine_submit_s16_2d(e: *mut same_engine, samples: *const i16, row_stride: u64, col_start: u64, n_cols: u32) -> c_int;
    // the reference's own item type: iter_events<I: IntoIterator<Item = f32>> (receiver.rs:119-130)
    pub fn same_engine_submit_f32(e: *mut same_engine, samples: *const f32, total_samples: u64, offsets: *const u64, lengths: *const u32) -> c_int;
    pub fn same_engine_submit_f32_device(e: *mut same_engine, d_samples: *const f32, total_samples: u64, offsets: *const u64,
                                         lengths: *const u32) -> c_int;
    pub fn same_engine_submit_zeros(e: *mut same_engine, lengths: *const u32) -> c_int;
    pub fn same_engine_lost_events(e: *mut same_engine, events_lost: *mut u64, payloads_lost: *mut u64) -> c_int;
    pub fn same_engine_sync(e: *mut same_engine) -> c_int;
    pub fn same_engine_pending(e: *mut same_engine, n_events: *mut usize, n_payload: *mut usize) -> c_int;
    pub fn same_engine_drain_events(e: *mut same_engine, events: *mut same_event, events_cap: usize, n_events: *mut usize,
                                    payload: *mut u8, payload_cap: usize, n_payload: *mut usize) -> c_int;
    pub fn same_host_alloc(bytes: usize) -> *mut c_void;
    pub fn same_host_free(p: *mut c_void);
    pub fn same_h2d_probe(device: c_int, host: *const c_void, row_stride_bytes: usize, width_bytes: usize, rows: usize, reps: c_int,
                          elapsed_ms: *mut f32) -> c_int;
    // samples already on the device (the engine's own corpus generator, or another CUDA producer)
    pub fn same_engine_submit_s16_device(e: *mut same_engine, d_samples: *const i16, total_samples: u64, offsets: *const u64,
                                         lengths: *const u32) -> c_int;
    pub fn same_engine_cuda_stream(e: *mut same_engine) -> *mut c_void;
    // SameReceiver: Clone  (used by flush() to stop at the sample of the first message)
    pub fn same_engine_snapshot(e: *mut same_engine, out: *mut *mut same_snapshot) -> c_int;
    pub fn same_engine_restore(e: *mut same_engine, snap: *const same_snapshot) -> c_int;
    pub fn same_snapshot_free(snap: *mut same_snapshot);
    // portable stream state (format in same_engine.h): SameReceiver: Clone for single streams, across engines/devices/processes
    pub fn same_engine_state_bytes(e: *const same_engine, n: u32) -> usize;
    pub fn same_engine_export_streams(e: *mut same_engine, ids: *const u32, n: u32, buf: *mut c_void, cap: usize,
                                      written: *mut usize) -> c_int;
    pub fn same_engine_import_streams(e: *mut same_engine, ids: *const u32, n: u32, buf: *const c_void, len: usize) -> c_int;
    pub fn same_state_info(buf: *const c_void, len: usize, cfg: *mut same_config, n_records: *mut u32) -> c_int;
    pub fn same_engine_set_event_capacity(e: *mut same_engine, max_events: usize, max_payload_bytes: usize) -> c_int;
    // diagnostics
    pub fn same_engine_enable_soft_trace(e: *mut same_engine, cap_per_stream: u32) -> c_int;
    pub fn same_engine_read_soft_trace(e: *mut same_engine, stream: u32, out: *mut same_soft_symbol, cap: usize, n: *mut usize) -> c_int;
    pub fn same_engine_set_option(e: *mut same_engine, key: *const c_char, value: c_int) -> c_int;
    pub fn same_engine_get_option(e: *mut same_engine, key: *const c_char, value: *mut c_int) -> c_int;
    pub fn same_engine_frontend_probe(e: *mut same_engine, d_samples: *const i16, total_samples: u64, offsets: *const u64,
                                      lengths: *const u32, reps: c_int, ms_per_launch: *mut f32) -> c_int;
    pub fn same_engine_last_timing(e: *mut same_engine, h2d_ms: *mut f32, kernel_ms: *mut f32) -> c_int;
    pub fn same_engine_launch_count(e: *const same_engine) -> u64;
    pub fn same_engine_timer_start(e: *mut same_engine) -> c_int;
    pub fn same_engine_timer_stop(e: *mut same_engine, elapsed_ms: *mut f32) -> c_int;
    pub fn same_engine_get_derived(e: *const same_engine, d: *mut same_derived, mark_re_im: *mut f32, space_re_im: *mut f32,
                                   cap_taps: usize) -> c_int;
    // one batch over several devices: one host thread + one engine per device inside the library
    pub fn same_multi_create(cfg: *const same_config, devices: *const c_int, n_devices: u32, n_streams: u32,
                             out: *mut *mut same_multi) -> c_int;
    pub fn same_multi_destroy(m: *mut same_multi);
    pub fn same_multi_last_error(m: *const same_multi) -> *const c_char;
    pub fn same_multi_num_shards(m: *const same_multi) -> u32;
    pub fn same_multi_num_streams(m: *const same_multi) -> u32;
    pub fn same_multi_shard_info(m: *const same_multi, shard: u32, device: *mut c_int, first_stream: *mut u32, n_streams: *mut u32) -> c_int;
    pub fn same_multi_engine(m: *mut same_multi, shard: u32) -> *mut same_engine;
    pub fn same_multi_submit_s16(m: *mut same_multi, samples: *const i16, total_samples: u64, offsets: *const u64, lengths: *const u32) -> c_int;
    pub fn same_multi_submit_f32(m: *mut same_multi, samples: *const f32, total_samples: u64, offsets: *const u64, lengths: *const u32) -> c_int;
    pub fn same_multi_submit_s16_2d(m: *mut same_multi, samples: *const i16, row_stride: u64, col_start: u64, n_cols: u32) -> c_int;
    pub fn same_multi_submit_zeros(m: *mut same_multi, lengths: *const u32) -> c_int;
    pub fn same_multi_sync(m: *mut same_multi) -> c_int;
    pub fn same_multi_reset(m: *mut same_multi) -> c_int;
    pub fn same_multi_input_sample_counters(m: *mut same_multi, out: *mut u64) -> c_int;
    pub fn same_multi_pending(m: *mut same_multi, n_events: *mut usize, n_payload: *mut usize) -> c_int;
    pub fn same_multi_drain_events(m: *mut same_multi, events: *mut same_event, events_cap: usize, n_events: *mut usize,
                                   payload: *mut u8, payload_cap: usize, n_payload: *mut usize) -> c_int;
    pub fn same_multi_state_bytes(m: *const same_multi, n: u32) -> usize;
    pub fn same_multi_export_streams(m: *mut same_multi, ids: *const u32, n: u32, buf: *mut c_void, cap: usize,
                                     written: *mut usize) -> c_int;
    pub fn same_multi_import_streams(m: *mut same_multi, ids: *const u32, n: u32, buf: *const c_void, len: usize) -> c_int;
}

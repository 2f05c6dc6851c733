//! `SameBatchReceiver`: the batched entry point next to `SameReceiver` (crates/sameold/src/receiver.rs:71-224).
//! Source only — not compiled in this repository (no Rust toolchain in the build image).
//!
//! It keeps the reference's surface: build from `SameReceiverBuilder`, feed audio, get `SameReceiverEvent`s /
//! `Message`s.  Decoding (link AND transport layer) happens in the CUDA engine; this file converts event records into
//! the crate's own types.  `Message` values are rebuilt with `Message::try_from((bytes, errs, bursts))`
//! (sameplace message.rs:718-736) from the header text and the parity / voting counts the engine reports.
use crate::ffi::*;
use crate::{LinkState, Message, MessageDecodeErr, MessageHeader, SameReceiverBuilder, TransportState};
use std::ptr;

/// `n_streams` receivers sharded over one or more CUDA devices of this box: one engine + one host thread per device
/// inside the native library (`same_multi_*`), no collective — streams are independent.
pub struct SameBatchReceiver {
    multi: *mut same_multi,
    n_streams: u32,
    devices: Vec<i32>,
}

/// One event of one stream, in order of occurrence per stream (== what `iter_events` yields on that stream).
pub struct BatchedEvent {
    pub stream: u32,
    pub input_sample_counter: u64,
    pub what: crate::SameEventType,
}

impl SameBatchReceiver {
    /// == `SameReceiverBuilder::build()` for `n_streams` receivers on CUDA device `device`.
    pub fn new(builder: &SameReceiverBuilder, n_streams: u32, device: i32) -> Result<Self, String> {
        Self::new_multi(builder, n_streams, &[device])
    }

    /// The same over several devices: stream i lives on `devices[i * devices.len() / n_streams]` (contiguous shards).
    pub fn new_multi(builder: &SameReceiverBuilder, n_streams: u32, devices: &[i32]) -> Result<Self, String> {
        let (unlocked, locked) = builder.timing_bandwidth();
        let (open, close) = builder.squelch_power();
        let eq = builder.adaptive_equalizer();
        let cfg = same_config {
            input_rate: builder.input_rate(),
            dc_blocker_len: builder.dc_blocker_length(),
            agc_bandwidth: builder.agc_bandwidth(),
            agc_gain_min: builder.agc_gain_limits()[0],
            agc_gain_max: builder.agc_gain_limits()[1],
            timing_bw_unlocked: unlocked,
            timing_bw_locked: locked,
            timing_max_deviation: builder.timing_max_deviation(),
            squelch_power_open: open,
            squelch_power_close: close,
            squelch_bandwidth: builder.squelch_bandwidth(),
            preamble_max_errors: builder.preamble_max_errors(),
            eq_enabled: eq.is_some() as u32,
            eq_nff: eq.map(|e| e.filter_order().0 as u32).unwrap_or(1),
            eq_nfb: eq.map(|e| e.filter_order().1 as u32).unwrap_or(1),
            eq_relaxation: eq.map(|e| e.relaxation()).unwrap_or(0.0),
            eq_regularization: eq.map(|e| e.regularization()).unwrap_or(1.0e-6),
            frame_prefix_max_errors: builder.frame_prefix_max_errors(),
            frame_max_invalid_bytes: builder.frame_max_invalid(),
        };
        Self::create(&cfg, n_streams, devices)
    }

    fn create(cfg: &same_config, n_streams: u32, devices: &[i32]) -> Result<Self, String> {
        let mut multi = ptr::null_mut();
        let rc = unsafe { same_multi_create(cfg, devices.as_ptr(), devices.len() as u32, n_streams, &mut multi) };
        if rc != 0 {
            let msg = unsafe { std::ffi::CStr::from_ptr(same_multi_last_error(ptr::null())) };
            return Err(format!("same_multi_create: {} ({})", rc, msg.to_string_lossy()));
        }
        Ok(Self { multi, n_streams, devices: devices.to_vec() })
    }

    /// The complete receiver state of streams `ids` (`None`: every stream, in order) as a portable buffer (format in
    /// same_engine.h) that any engine with the same configuration can import, on any device or in another process.
    pub fn export_streams(&mut self, ids: Option<&[u32]>) -> Result<Vec<u8>, String> {
        let n = ids.map(|v| v.len() as u32).unwrap_or(self.n_streams);
        let ids_ptr = ids.map(|v| v.as_ptr()).unwrap_or(ptr::null());
        let mut buf = vec![0u8; unsafe { same_multi_state_bytes(self.multi, n) }];
        let mut written = 0usize;
        unsafe {
            check(self.multi, same_multi_export_streams(self.multi, ids_ptr, n, buf.as_mut_ptr() as *mut _, buf.len(), &mut written))?;
        }
        Ok(buf)
    }

    /// Record i -> stream `ids[i]` (`None`: record i -> stream i): like `reset` of those streams followed by writing the
    /// recorded state; all or nothing.
    pub fn import_streams(&mut self, data: &[u8], ids: Option<&[u32]>) -> Result<(), String> {
        let n = match ids {
            Some(v) => v.len() as u32,
            None => state_info(data)?.1,
        };
        let ids_ptr = ids.map(|v| v.as_ptr()).unwrap_or(ptr::null());
        unsafe { check(self.multi, same_multi_import_streams(self.multi, ids_ptr, n, data.as_ptr() as *const _, data.len())) }
    }

    /// A new receiver batch on `devices`, built from the configuration embedded in `data` and holding every record.
    pub fn from_state(data: &[u8], devices: &[i32]) -> Result<Self, String> {
        let (cfg, n) = state_info(data)?;
        let mut rx = Self::create(&cfg, n, devices)?;
        rx.import_streams(data, None)?;
        Ok(rx)
    }

    /// == `iter_events(chunk)` driven to exhaustion on every stream.  `chunks[i]` is stream i's next s16 samples
    /// (the reference takes `sa as f32`, crates/samedec/src/app.rs:112; the engine ingests the i16 directly).
    pub fn process(&mut self, chunks: &[&[i16]]) -> Result<Vec<BatchedEvent>, String> {
        assert_eq!(chunks.len(), self.n_streams as usize);
        let mut flat = Vec::with_capacity(chunks.iter().map(|c| c.len()).sum());
        let (mut offsets, mut lengths) = (Vec::new(), Vec::new());
        for c in chunks {
            offsets.push(flat.len() as u64);
            lengths.push(c.len() as u32);
            flat.extend_from_slice(c);
        }
        unsafe {
            check(self.multi, same_multi_submit_s16(self.multi, flat.as_ptr(), flat.len() as u64, offsets.as_ptr(), lengths.as_ptr()))?;
            check(self.multi, same_multi_sync(self.multi))?;
        }
        self.drain()
    }

    /// The reference's own item type: `iter_events<I: IntoIterator<Item = f32>>` (receiver.rs:119-130), any scale.
    pub fn process_f32(&mut self, chunks: &[&[f32]]) -> Result<Vec<BatchedEvent>, String> {
        assert_eq!(chunks.len(), self.n_streams as usize);
        let mut flat = Vec::with_capacity(chunks.iter().map(|c| c.len()).sum());
        let (mut offsets, mut lengths) = (Vec::new(), Vec::new());
        for c in chunks {
            offsets.push(flat.len() as u64);
            lengths.push(c.len() as u32);
            flat.extend_from_slice(c);
        }
        unsafe {
            check(self.multi, same_multi_submit_f32(self.multi, flat.as_ptr(), flat.len() as u64, offsets.as_ptr(), lengths.as_ptr()))?;
            check(self.multi, same_multi_sync(self.multi))?;
        }
        self.drain()
    }

    /// == `iter_messages` for every stream: `(stream, Message)` in order of occurrence per stream.
    pub fn iter_messages_batched(&mut self, chunks: &[&[i16]]) -> Result<Vec<(u32, Message)>, String> {
        Ok(self
            .process(chunks)?
            .into_iter()
            .filter_map(|e| match e.what {
                crate::SameEventType::Transport(TransportState::Message(Ok(m))) => Some((e.stream, m)),
                _ => None,
            })
            .collect())
    }

    fn drain(&mut self) -> Result<Vec<BatchedEvent>, String> {
        let (mut nev, mut npay) = (0usize, 0usize);
        unsafe { check(self.multi, same_multi_pending(self.multi, &mut nev, &mut npay))? };
        let mut evs = vec![same_event::default(); nev];
        let mut pay = vec![0u8; npay.max(1)];
        unsafe {
            check(self.multi, same_multi_drain_events(self.multi, evs.as_mut_ptr(), nev, &mut nev, pay.as_mut_ptr(), pay.len(), &mut npay))?;
        }
        Ok(evs
            .iter()
            .map(|e| {
                let data = &pay[e.data_offset as usize..(e.data_offset + e.data_len.min(1024)) as usize];
                let what = match e.kind {
                    SAME_EV_LINK_NOCARRIER => LinkState::NoCarrier.into(),
                    SAME_EV_LINK_SEARCHING => LinkState::Searching.into(),
                    SAME_EV_LINK_READING => LinkState::Reading.into(),
                    SAME_EV_LINK_BURST => LinkState::Burst(data.to_vec()).into(),
                    SAME_EV_TR_IDLE => TransportState::Idle.into(),
                    SAME_EV_TR_ASSEMBLING => TransportState::Assembling.into(),
                    SAME_EV_TR_MSG_EOM => TransportState::Message(Ok(Message::EndOfMessage)).into(),
                    SAME_EV_TR_MSG_SOM => {
                        // rebuild per-byte arrays that sum to the engine's counts (message.rs:209-254)
                        let n = data.len();
                        let mut errs = vec![0u8; n];
                        let mut left = e.parity_errors as usize;
                        for b in errs.iter_mut() { let t = left.min(255); *b = t as u8; left -= t; }
                        let mut bursts = vec![2u8; n];
                        for b in bursts.iter_mut().take(e.voting_bytes as usize) { *b = 3; }
                        let hdr = MessageHeader::new_with_error_info(String::from_utf8_lossy(data).into_owned(), &errs, &bursts)
                            .expect("engine emitted a header that fails sameplace validation");
                        TransportState::Message(Ok(Message::StartOfMessage(hdr))).into()
                    }
                    _ => TransportState::Message(Err(match e.err {
                        1 => MessageDecodeErr::UnrecognizedPrefix,
                        2 => MessageDecodeErr::NotAscii,
                        _ => MessageDecodeErr::Malformed,
                    }))
                    .into(),
                };
                BatchedEvent { stream: e.stream, input_sample_counter: e.input_sample_counter, what }
            })
            .collect())
    }
}

/// == `SameReceiver: Clone` (receiver.rs:70): an independent batch on the same devices in the same state.
impl Clone for SameBatchReceiver {
    fn clone(&self) -> Self {
        let mut me = Self { multi: self.multi, n_streams: self.n_streams, devices: Vec::new() };
        let data = me.export_streams(None);
        std::mem::forget(me);   // borrowed handle: not ours to destroy
        Self::from_state(&data.expect("exporting the receiver state failed"), &self.devices)
            .expect("importing the receiver state failed")
    }
}

/// (configuration, number of records) of an export buffer: header checks only.
pub fn state_info(data: &[u8]) -> Result<(same_config, u32), String> {
    let mut cfg = std::mem::MaybeUninit::<same_config>::zeroed();
    let mut n = 0u32;
    let rc = unsafe { same_state_info(data.as_ptr() as *const _, data.len(), cfg.as_mut_ptr(), &mut n) };
    if rc != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(same_last_error()) };
        return Err(format!("same_state_info: {} ({})", rc, msg.to_string_lossy()));
    }
    Ok((unsafe { cfg.assume_init() }, n))
}

impl Drop for SameBatchReceiver {
    fn drop(&mut self) {
        unsafe { same_multi_destroy(self.multi) }
    }
}

unsafe fn check(m: *mut same_multi, rc: i32) -> Result<(), String> {
    if rc == 0 {
        Ok(())
    } else {
        Err(format!("same_engine error {}: {}", rc, std::ffi::CStr::from_ptr(same_multi_last_error(m)).to_string_lossy()))
    }
}

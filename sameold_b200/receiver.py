"""Host-side mirror of the reference's receiver API over the C ABI (include/same_engine.h).

Same names, argument meaning and error behaviour as the Rust surface it stands in for (the Rust toolchain is absent
here; bindings/rust/ holds the uncompiled Rust source of the same layer):

    SameReceiverBuilder / EqualizerBuilder    crates/sameold/src/receiver/builder.rs:50-279, 369-425
    SameReceiver.iter_events / iter_messages / input_rate / input_sample_counter / reset / flush
                                              crates/sameold/src/receiver.rs:119-224
    SameReceiverEvent / LinkState / TransportState / Message
                                              crates/sameold/src/receiver/output.rs, crates/sameplace/src/message.rs:62-98

plus the batched entry point the north star asks for: SameBatchReceiver.process / iter_messages_batched /
decode_samedec.  All decoding happens in the CUDA engine; this module only moves buffers and turns event records into
objects.
"""
import ctypes as C
from dataclasses import dataclass
from typing import Iterable, Iterator, List, Optional, Sequence

import numpy as np

from . import _lib

# ---------------------------------------------------------------------------------------------------------------------
# Event model (output.rs)
# ---------------------------------------------------------------------------------------------------------------------
EV_LINK_NOCARRIER, EV_LINK_SEARCHING, EV_LINK_READING, EV_LINK_BURST = 0, 1, 2, 3
EV_TR_IDLE, EV_TR_ASSEMBLING, EV_TR_MSG_SOM, EV_TR_MSG_EOM, EV_TR_MSG_ERR = 16, 17, 18, 19, 20

_DECODE_ERR = {
    1: "invalid SAME header: unrecognized prefix",            # MessageDecodeErr::UnrecognizedPrefix  message.rs:88
    2: "invalid SAME header: message contains non-ASCII characters",  # NotAscii           message.rs:92
    3: "invalid SAME header: message text does not match required pattern",  # Malformed   message.rs:96
}
_KIND_NAMES = {
    0: "LinkState::NoCarrier", 1: "LinkState::Searching", 2: "LinkState::Reading", 3: "LinkState::Burst",
    16: "TransportState::Idle", 17: "TransportState::Assembling", 18: "TransportState::Message(Ok(StartOfMessage))",
    19: "TransportState::Message(Ok(EndOfMessage))", 20: "TransportState::Message(Err)",
}


class SameEngineError(RuntimeError):
    """A non-zero status from the C ABI (resource/engine errors; decode errors are event values, never exceptions)."""

    def __init__(self, code, text):
        super().__init__(f"same_engine error {code}: {text}")
        self.code = code


@dataclass(frozen=True)
class Message:
    """== sameold::Message (sameplace message.rs:62-83): StartOfMessage(header) | EndOfMessage."""

    text: str
    is_start: bool
    parity_error_count: int = 0   # message.rs:123
    voting_byte_count: int = 0    # message.rs:140

    def as_str(self) -> str:      # message.rs:105
        return self.text

    def __str__(self):
        return self.text


@dataclass(frozen=True)
class SameReceiverEvent:
    """== SameReceiverEvent (output.rs:24-27) + the stream it came from."""

    stream: int
    kind: int
    sample: int                   # input_sample_counter()  output.rs:111
    symbol_count: int             # diagnostic
    data: bytes = b""             # burst bytes or message text
    err: int = 0
    parity_errors: int = 0
    voting_bytes: int = 0
    flags: int = 0

    def what(self) -> str:
        return _KIND_NAMES.get(self.kind, str(self.kind))

    def input_sample_counter(self) -> int:
        return self.sample

    def is_link(self) -> bool:
        return self.kind < 16

    def burst(self) -> Optional[bytes]:            # output.rs:70-75
        return self.data if self.kind == EV_LINK_BURST else None

    def message_ok(self) -> Optional[Message]:     # output.rs:58-63
        if self.kind == EV_TR_MSG_SOM:
            return Message(self.data.decode("ascii"), True, self.parity_errors, self.voting_bytes)
        if self.kind == EV_TR_MSG_EOM:
            return Message("NNNN", False)
        return None

    def message_err(self) -> Optional[str]:
        return _DECODE_ERR.get(self.err) if self.kind == EV_TR_MSG_ERR else None

    def into_message_ok(self) -> Optional[Message]:  # output.rs:99-104
        return self.message_ok()

    def key(self):
        """The fields that must match the oracle bit for bit."""
        return (self.kind, self.err, self.sample, self.symbol_count, self.data, self.parity_errors, self.voting_bytes)

    def __repr__(self):
        return f"<s{self.stream} {self.what()} @{self.sample} sym {self.symbol_count} {self.data[:40]!r}>"


# ---------------------------------------------------------------------------------------------------------------------
# Builders (builder.rs)
# ---------------------------------------------------------------------------------------------------------------------
def _f32(x):
    return float(np.float32(x))


def _clamp(x, lo, hi):  # f32::clamp
    x = _f32(x)
    if x < lo:
        x = lo
    if x > hi:
        x = hi
    return x


class EqualizerBuilder:
    """== EqualizerBuilder (builder.rs:360-437)."""

    def __init__(self):
        self.nfeedforward, self.nfeedback = 6, 4
        self._relaxation, self._regularization = _f32(0.05), _f32(1.0e-6)

    def with_filter_order(self, nfeedforward: int, nfeedback: int) -> "EqualizerBuilder":  # builder.rs:393-397
        self.nfeedforward = max(int(nfeedforward), 1)
        self.nfeedback = min(max(int(nfeedback), 1), self.nfeedforward)
        return self

    def with_relaxation(self, relaxation: float) -> "EqualizerBuilder":  # builder.rs:404-407
        self._relaxation = _clamp(relaxation, 0.0, 1.0)
        return self

    def with_regularization(self, regularization: float) -> "EqualizerBuilder":  # builder.rs:416-419
        self._regularization = _clamp(regularization, 0.0, float(np.finfo(np.float32).max))
        return self

    def filter_order(self):
        return (self.nfeedforward, self.nfeedback)

    def relaxation(self):
        return self._relaxation

    def regularization(self):
        return self._regularization


class SameReceiverBuilder:
    """== SameReceiverBuilder (builder.rs:14-357).  `SameReceiverBuilder(22050)` == `SameReceiverBuilder::new(22050)`."""

    def __init__(self, input_rate: int = 22050):
        lib = _lib.load()
        self._cfg = _lib.SameConfig()
        lib.same_config_default(C.byref(self._cfg), int(input_rate))

    @classmethod
    def new(cls, input_rate: int) -> "SameReceiverBuilder":
        return cls(input_rate)

    @classmethod
    def samedec(cls, input_rate: int = 22050) -> "SameReceiverBuilder":
        """The builder `samedec` constructs (crates/samedec/src/main.rs:29-37)."""
        b = cls(input_rate)
        _lib.load().same_config_samedec(C.byref(b._cfg), int(input_rate))
        return b

    # --- setters, same clamping as the reference ---
    def with_dc_blocker_length(self, length: float):                       # builder.rs:95-98
        self._cfg.dc_blocker_len = max(0.0, _f32(length)); return self

    def with_agc_bandwidth(self, bw: float):                               # builder.rs:107-110
        self._cfg.agc_bandwidth = _clamp(bw, 0.0, 1.0); return self

    def with_agc_gain_limits(self, gmin: float, gmax: float):              # builder.rs:122-125
        self._cfg.agc_gain_min, self._cfg.agc_gain_max = _f32(gmin), _f32(gmax); return self

    def with_timing_bandwidth(self, unlocked_bw: float, locked_bw: float):  # builder.rs:143-147
        self._cfg.timing_bw_unlocked = _clamp(unlocked_bw, 0.0, 1.0)
        self._cfg.timing_bw_locked = _clamp(locked_bw, 0.0, self._cfg.timing_bw_unlocked); return self

    def with_timing_max_deviation(self, max_dev: float):                   # builder.rs:162-165
        self._cfg.timing_max_deviation = _clamp(max_dev, 0.0, 0.5); return self

    def with_squelch_power(self, power_open: float, power_close: float):   # builder.rs:190-194
        self._cfg.squelch_power_open = _clamp(power_open, 0.0, 1.0)
        self._cfg.squelch_power_close = min(_f32(power_close), _f32(power_open)); return self

    def with_squelch_bandwidth(self, bw: float):                           # builder.rs:203-206
        self._cfg.squelch_bandwidth = _f32(bw); return self

    def with_preamble_max_errors(self, max_err: int):                      # builder.rs:218-221
        self._cfg.preamble_max_errors = int(max_err); return self

    def with_adaptive_equalizer(self, eql: EqualizerBuilder):              # builder.rs:229-232
        self._cfg.eq_enabled = 1
        self._cfg.eq_nff, self._cfg.eq_nfb = eql.nfeedforward, eql.nfeedback
        self._cfg.eq_relaxation, self._cfg.eq_regularization = eql.relaxation(), eql.regularization(); return self

    def without_adaptive_equalizer(self):                                  # builder.rs:239-242
        self._cfg.eq_enabled = 0; return self

    def with_frame_prefix_max_errors(self, max_err: int):                  # builder.rs:256-259
        self._cfg.frame_prefix_max_errors = min(max(int(max_err), 0), 7); return self

    def with_frame_max_invalid(self, max_invalid: int):                    # builder.rs:277-280
        self._cfg.frame_max_invalid_bytes = int(max_invalid); return self

    # --- getters ---
    def input_rate(self): return self._cfg.input_rate
    def dc_blocker_length(self): return self._cfg.dc_blocker_len
    def agc_bandwidth(self): return self._cfg.agc_bandwidth
    def agc_gain_limits(self): return (self._cfg.agc_gain_min, self._cfg.agc_gain_max)
    def timing_bandwidth(self): return (self._cfg.timing_bw_unlocked, self._cfg.timing_bw_locked)
    def timing_max_deviation(self): return self._cfg.timing_max_deviation
    def squelch_power(self): return (self._cfg.squelch_power_open, self._cfg.squelch_power_close)
    def squelch_bandwidth(self): return self._cfg.squelch_bandwidth
    def preamble_max_errors(self): return self._cfg.preamble_max_errors
    def frame_prefix_max_errors(self): return self._cfg.frame_prefix_max_errors
    def frame_max_invalid(self): return self._cfg.frame_max_invalid_bytes

    def adaptive_equalizer(self) -> Optional[EqualizerBuilder]:
        if not self._cfg.eq_enabled:
            return None
        e = EqualizerBuilder()
        e.nfeedforward, e.nfeedback = self._cfg.eq_nff, self._cfg.eq_nfb
        e._relaxation, e._regularization = self._cfg.eq_relaxation, self._cfg.eq_regularization
        return e

    def config(self) -> "_lib.SameConfig":
        c = _lib.SameConfig()
        C.memmove(C.byref(c), C.byref(self._cfg), C.sizeof(c))
        return c

    # --- build ---
    def build(self, device: int = 0) -> "SameReceiver":
        """== SameReceiverBuilder::build (builder.rs:81-84): one receiver (an engine with a single stream)."""
        return SameReceiver(SameBatchReceiver(self.config(), 1, device))

    def build_batch(self, n_streams: int, device: int = 0) -> "SameBatchReceiver":
        """The batched entry point: n_streams independent receivers resident on one GPU."""
        return SameBatchReceiver(self.config(), n_streams, device)

    def build_multi(self, n_streams: int, devices: Sequence[int]) -> "SameMultiReceiver":
        """n_streams receivers sharded over several GPUs of this box (one host thread + engine per device)."""
        return SameMultiReceiver(self.config(), n_streams, devices)


# ---------------------------------------------------------------------------------------------------------------------
# Batched receiver
# ---------------------------------------------------------------------------------------------------------------------
class SameBatchReceiver:
    """N independent SameReceivers on one CUDA device; state persists across calls (chunked == whole, bit-exact)."""

    def __init__(self, cfg, n_streams: int, device: int = 0):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self._cfg = cfg
        rc = self._lib.same_engine_create(C.byref(cfg), int(device), int(n_streams), C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            raise SameEngineError(rc, self._lib.same_last_error().decode())
        self.n_streams = int(n_streams)
        self.device = int(device)

    # -- plumbing --
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.same_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise SameEngineError(rc, self._lib.same_engine_last_error(self._h).decode())

    @property
    def handle(self):
        return self._h

    def input_rate(self) -> int:                                # receiver.rs:167
        return self._lib.same_engine_input_rate(self._h)

    def input_sample_counters(self) -> np.ndarray:              # receiver.rs:175
        out = np.zeros(self.n_streams, np.uint64)
        self._ck(self._lib.same_engine_input_sample_counters(self._h, out.ctypes.data))
        return out

    def reset(self, stream_ids: Optional[Sequence[int]] = None):  # receiver.rs:182-198
        if stream_ids is None:
            self._ck(self._lib.same_engine_reset(self._h, None, 0))
        else:
            ids = np.ascontiguousarray(stream_ids, dtype=np.uint32)
            self._ck(self._lib.same_engine_reset(self._h, ids.ctypes.data, ids.size))

    def set_event_capacity(self, max_events: int, max_payload_bytes: int):
        self._ck(self._lib.same_engine_set_event_capacity(self._h, max_events, max_payload_bytes))

    def derived(self):
        d = _lib.SameDerived()
        self._ck(self._lib.same_engine_get_derived(self._h, C.byref(d), None, None, 0))
        mark = np.zeros((d.ntaps, 2), np.float32)
        space = np.zeros((d.ntaps, 2), np.float32)
        self._ck(self._lib.same_engine_get_derived(self._h, C.byref(d), mark.ctypes.data, space.ctypes.data, d.ntaps))
        out = {n: getattr(d, n) for n, _ in _lib.SameDerived._fields_}
        out["mark"], out["space"] = mark, space
        return out

    # -- submit / drain --
    @staticmethod
    def _pack(chunks) -> "tuple[np.ndarray, np.ndarray, np.ndarray]":
        """list of 1-D int16 arrays (ragged, None/empty = no input) or a 2-D array -> (flat, offsets, lengths)."""
        if isinstance(chunks, np.ndarray) and chunks.ndim == 2:
            a = np.ascontiguousarray(chunks, dtype=np.int16)
            n, m = a.shape
            return a.reshape(-1), np.arange(n, dtype=np.uint64) * np.uint64(m), np.full(n, m, np.uint32)
        arrs = [np.zeros(0, np.int16) if c is None else np.ascontiguousarray(c, dtype=np.int16).reshape(-1) for c in chunks]
        lengths = np.array([a.size for a in arrs], np.uint32)
        offsets = np.zeros(len(arrs), np.uint64)
        if len(arrs) > 1:
            offsets[1:] = np.cumsum(lengths[:-1], dtype=np.uint64)
        flat = np.concatenate(arrs) if arrs else np.zeros(0, np.int16)
        return flat, offsets, lengths

    def submit(self, chunks):
        """Feed one chunk per stream (host memory).  Asynchronous; keep nothing — the data is staged before return only
        if pageable (numpy) memory is used, so this wrapper syncs before dropping its packed copy in `process`."""
        flat, offsets, lengths = self._pack(chunks)
        if lengths.size != self.n_streams:
            raise ValueError(f"expected {self.n_streams} chunks, got {lengths.size}")
        self._keep = (flat, offsets, lengths)
        self._ck(self._lib.same_engine_submit_s16(self._h, flat.ctypes.data, flat.size, offsets.ctypes.data, lengths.ctypes.data))

    def submit_f32(self, chunks):
        """Feed one chunk of f32 samples per stream — the reference's own item type (receiver.rs:119-130; lib.rs:78-79:
        any scale, the AGC normalises).  Takes the literal f32 DC-blocker recursion (rate-generic kernel)."""
        if isinstance(chunks, np.ndarray) and chunks.ndim == 2:
            arrs = [np.ascontiguousarray(r, dtype=np.float32) for r in chunks]
        else:
            arrs = [np.zeros(0, np.float32) if c is None else np.ascontiguousarray(c, dtype=np.float32).reshape(-1) for c in chunks]
        if len(arrs) != self.n_streams:
            raise ValueError(f"expected {self.n_streams} chunks, got {len(arrs)}")
        lengths = np.array([a.size for a in arrs], np.uint32)
        offsets = np.zeros(len(arrs), np.uint64)
        if len(arrs) > 1:
            offsets[1:] = np.cumsum(lengths[:-1], dtype=np.uint64)
        flat = np.concatenate(arrs) if arrs else np.zeros(0, np.float32)
        self._keep = (flat, offsets, lengths)
        self._ck(self._lib.same_engine_submit_f32(self._h, flat.ctypes.data, flat.size, offsets.ctypes.data, lengths.ctypes.data))

    def process_f32(self, chunks) -> List[List[SameReceiverEvent]]:
        self.submit_f32(chunks)
        self.sync()
        return self.drain_by_stream()

    def lost_events(self):
        """(events dropped, payloads dropped) because an arena was full, since create."""
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._lib.same_engine_lost_events(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def submit_flat(self, flat: np.ndarray, offsets: np.ndarray, lengths: np.ndarray):
        """Zero-copy variant: caller-owned flat int16 buffer (e.g. pinned) + per-stream offsets/lengths."""
        assert flat.dtype == np.int16 and offsets.dtype == np.uint64 and lengths.dtype == np.uint32
        self._keep = (flat, offsets, lengths)
        self._ck(self._lib.same_engine_submit_s16(self._h, flat.ctypes.data, flat.size, offsets.ctypes.data, lengths.ctypes.data))

    def submit_2d(self, host_ptr: int, row_stride: int, col_start: int, n_cols: int):
        """Time slice [col_start, col_start+n_cols) of a host matrix int16[n_streams][row_stride] (raw host pointer,
        ideally pinned memory from same_host_alloc): one strided copy, overlapped with the previous chunk's kernel."""
        self._ck(self._lib.same_engine_submit_s16_2d(self._h, C.c_void_p(host_ptr), int(row_stride), int(col_start), int(n_cols)))

    def submit_device(self, d_ptr: int, total_samples: int, offsets: np.ndarray, lengths: np.ndarray):
        """Samples already resident in this device's memory (raw device pointer, e.g. torch_tensor.data_ptr())."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        self._keep = (offsets, lengths)
        self._ck(self._lib.same_engine_submit_s16_device(self._h, C.c_void_p(d_ptr), int(total_samples), offsets.ctypes.data, lengths.ctypes.data))

    def submit_zeros(self, lengths):
        lengths = np.ascontiguousarray(np.broadcast_to(np.asarray(lengths, dtype=np.uint32), (self.n_streams,)))
        self._keep = (lengths,)
        self._ck(self._lib.same_engine_submit_zeros(self._h, lengths.ctypes.data))

    def sync(self):
        self._ck(self._lib.same_engine_sync(self._h))
        self._keep = None

    def drain(self) -> List[SameReceiverEvent]:
        """All pending events, sorted by (stream, order of occurrence)."""
        nev, npay = C.c_size_t(), C.c_size_t()
        self._ck(self._lib.same_engine_pending(self._h, C.byref(nev), C.byref(npay)))
        self._keep = None
        if nev.value == 0:
            return []
        evs = (_lib.SameEvent * nev.value)()
        pay = (C.c_uint8 * max(npay.value, 1))()
        self._ck(self._lib.same_engine_drain_events(self._h, evs, nev.value, C.byref(nev), pay, max(npay.value, 1), C.byref(npay)))
        payload = bytes(pay[: npay.value])
        out = []
        for e in evs[: nev.value]:
            n = min(e.data_len, 1024) if e.kind == EV_LINK_BURST else e.data_len
            out.append(SameReceiverEvent(e.stream, e.kind, e.input_sample_counter, e.symbol_count,
                                         payload[e.data_offset: e.data_offset + n], e.err, e.parity_errors,
                                         e.voting_bytes, e.flags))
        return out

    @staticmethod
    def events_from_raw(evs: np.ndarray, pay: np.ndarray) -> List[SameReceiverEvent]:
        """same_event records (drain_raw) -> SameReceiverEvent objects."""
        payload = pay.tobytes()
        out = []
        for e in evs:
            n = min(int(e["data_len"]), 1024) if e["kind"] == EV_LINK_BURST else int(e["data_len"])
            o = int(e["data_offset"])
            out.append(SameReceiverEvent(int(e["stream"]), int(e["kind"]), int(e["sample"]), int(e["symbol_count"]),
                                         payload[o:o + n], int(e["err"]), int(e["parity_errors"]),
                                         int(e["voting_bytes"]), int(e["flags"])))
        return out

    EVENT_DTYPE = np.dtype([("stream", "<u4"), ("seq", "<u4"), ("sample", "<u8"), ("symbol_count", "<u8"),
                            ("kind", "<u4"), ("err", "<u4"), ("data_offset", "<u4"), ("data_len", "<u4"),
                            ("parity_errors", "<u2"), ("voting_bytes", "<u2"), ("flags", "<u4")])

    def drain_raw(self, reuse: bool = False):
        """All pending events as a numpy structured array (same_event records, sorted by stream then occurrence) plus
        the payload arena — no per-event Python objects (what a high-rate consumer uses).  `reuse=True` returns views
        into buffers owned by the receiver (valid until the next drain): no allocation, no page faults per call."""
        nev, npay = C.c_size_t(), C.c_size_t()
        self._ck(self._lib.same_engine_pending(self._h, C.byref(nev), C.byref(npay)))
        self._keep = None
        if reuse:
            if getattr(self, "_raw_ev", None) is None or self._raw_ev.size < nev.value:
                self._raw_ev = np.empty(max(nev.value, 1) * 5 // 4 + 1024, self.EVENT_DTYPE)
            if getattr(self, "_raw_pay", None) is None or self._raw_pay.size < npay.value:
                self._raw_pay = np.empty(max(npay.value, 1) * 5 // 4 + 4096, np.uint8)
            evs, pay = self._raw_ev, self._raw_pay
        else:
            evs = np.empty(nev.value, self.EVENT_DTYPE)
            pay = np.empty(max(npay.value, 1), np.uint8)
        if nev.value:
            self._ck(self._lib.same_engine_drain_events(self._h, evs.ctypes.data, evs.size, C.byref(nev), pay.ctypes.data,
                                                        pay.size, C.byref(npay)))
        return evs[: nev.value], pay[: npay.value]

    def drain_by_stream(self) -> List[List[SameReceiverEvent]]:
        out: List[List[SameReceiverEvent]] = [[] for _ in range(self.n_streams)]
        for e in self.drain():
            out[e.stream].append(e)
        return out

    # -- the batched entry points --
    def process(self, chunks) -> List[List[SameReceiverEvent]]:
        """== iter_events(chunk) driven to exhaustion on every stream; returns the events per stream."""
        self.submit(chunks)
        self.sync()
        return self.drain_by_stream()

    def iter_events_batched(self, chunks) -> Iterator[SameReceiverEvent]:
        for evs in self.process(chunks):
            yield from evs

    def iter_messages_batched(self, chunks) -> Iterator["tuple[int, Message]"]:
        """== iter_messages (receiver.rs:155-161) for every stream: yields (stream, Message)."""
        for e in self.iter_events_batched(chunks):
            m = e.message_ok()
            if m is not None:
                yield (e.stream, m)

    def flush_samedec(self) -> List[List[SameReceiverEvent]]:
        """samedec's end-of-input rule (crates/samedec/src/app.rs:71-74,103-119): flush() = up to 4 s of zeros,
        abandoned at the first message, repeated until a whole 4 s of zeros yields no message.  Returns the events
        that rule lets through, per stream.  (Equivalent: feed zeros; stop input_rate*4 zeros after the last message.)"""
        nflush = self.input_rate() * 4
        out: List[List[SameReceiverEvent]] = [[] for _ in range(self.n_streams)]
        pos = self.input_sample_counters().astype(np.int64)
        origin = pos.copy()                 # sample counter at which each stream's current flush() began
        active = np.ones(self.n_streams, bool)
        while active.any():
            # run every active stream to the end of its current flush window (origin + 4 s)
            lens = np.where(active, origin + nflush - pos, 0).astype(np.uint32)
            self.submit_zeros(lens)
            self.sync()
            evs = self.drain_by_stream()
            pos = pos + lens
            for s in range(self.n_streams):
                if not active[s]:
                    continue
                out[s].extend(evs[s])
                msgs = [e.sample for e in evs[s] if e.message_ok() is not None]
                if msgs:
                    origin[s] = msgs[-1]    # flush() returned there; the next flush() starts a fresh 4 s window
                else:
                    active[s] = False       # a whole window without a message: the app loop ends (app.rs:72)
        return out

    def decode_samedec(self, recordings) -> List[List[str]]:
        """What `samedec --file F` prints for each recording (one str per message line): whole input, then the EOF
        flush rule.  Streams must be freshly built or reset."""
        evs = self.process(recordings)
        tail = self.flush_samedec()
        return [[str(e.message_ok()) for e in (a + b) if e.message_ok() is not None] for a, b in zip(evs, tail)]

    # -- diagnostics --
    def enable_soft_trace(self, cap_per_stream: int):
        self._ck(self._lib.same_engine_enable_soft_trace(self._h, int(cap_per_stream)))

    def read_soft_trace(self, stream: int) -> np.ndarray:
        n = C.c_size_t()
        self._ck(self._lib.same_engine_read_soft_trace(self._h, stream, None, 0, C.byref(n)))
        arr = (_lib.SameSoftSymbol * max(n.value, 1))()
        self._ck(self._lib.same_engine_read_soft_trace(self._h, stream, arr, n.value, C.byref(n)))
        a = np.frombuffer(arr, dtype=np.dtype([("sample", "<u8"), ("zero", "<f4"), ("sym", "<f4")]))[: n.value]
        return a.copy()

    def set_option(self, key: str, value: int):
        self._ck(self._lib.same_engine_set_option(self._h, key.encode(), int(value)))

    def frontend_probe(self, d_ptr: int, total_samples: int, offsets: np.ndarray, lengths: np.ndarray, reps: int = 5) -> float:
        """ms per launch of the front-end kernel alone on device-resident samples (measurement aid)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        ms = C.c_float()
        self._ck(self._lib.same_engine_frontend_probe(self._h, C.c_void_p(d_ptr), int(total_samples), offsets.ctypes.data,
                                                      lengths.ctypes.data, int(reps), C.byref(ms)))
        return ms.value

    def get_option(self, key: str) -> int:
        v = C.c_int()
        self._ck(self._lib.same_engine_get_option(self._h, key.encode(), C.byref(v)))
        return v.value

    def last_timing(self):
        h2d, k = C.c_float(), C.c_float()
        self._ck(self._lib.same_engine_last_timing(self._h, C.byref(h2d), C.byref(k)))
        return h2d.value, k.value

    def timer_start(self):
        self._ck(self._lib.same_engine_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self._ck(self._lib.same_engine_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return self._lib.same_engine_launch_count(self._h)

    def snapshot(self):
        s = C.c_void_p()
        self._ck(self._lib.same_engine_snapshot(self._h, C.byref(s)))
        return s

    def restore(self, snap):
        self._ck(self._lib.same_engine_restore(self._h, snap))

    def free_snapshot(self, snap):
        self._lib.same_snapshot_free(snap)

    # -- portable stream state (format: include/same_engine.h) --
    def export_streams(self, ids: Optional[Sequence[int]] = None) -> bytes:
        """The complete receiver state of streams `ids` (None: all, in order) as a self-describing buffer that any
        engine with the same configuration can import, on any device or in another process.  Changes nothing."""
        return _export(self._lib, self._lib.same_engine_state_bytes, self._lib.same_engine_export_streams, self._h, ids,
                       self.n_streams, self._ck)

    def import_streams(self, data, ids: Optional[Sequence[int]] = None):
        """Record i -> stream ids[i] (None: record i -> stream i).  Like reset(ids) followed by writing the recorded
        state; all or nothing."""
        _import(self._lib.same_engine_import_streams, self._h, data, ids, self._ck)

    @classmethod
    def from_state(cls, data, device: int = 0) -> "SameBatchReceiver":
        """A new engine built from the configuration embedded in `data`, holding every record of it."""
        cfg, n = state_info(data)
        rx = cls(cfg, n, device)
        rx.import_streams(data)
        return rx


def _buffer(data) -> np.ndarray:
    """bytes / bytearray / memoryview / uint8 array -> a uint8 view (no copy)."""
    return np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data.reshape(-1).view(np.uint8)


def _ids(ids):
    if ids is None:
        return None, None
    a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1)
    return a, a.ctypes.data


def _export(lib, state_bytes, export, h, ids, n_streams, ck) -> bytes:
    a, p = _ids(ids)
    n = n_streams if a is None else a.size
    out = bytearray(state_bytes(h, n))
    written = C.c_size_t()
    cbuf = (C.c_char * len(out)).from_buffer(out)
    ck(export(h, p, n, C.addressof(cbuf), len(out), C.byref(written)))
    del cbuf
    return bytes(out)


def _import(imp, h, data, ids, ck):
    buf = _buffer(data)
    a, p = _ids(ids)
    n = state_info(buf)[1] if a is None else a.size
    ck(imp(h, p, n, buf.ctypes.data, buf.size))


def state_info(data) -> "tuple[_lib.SameConfig, int]":
    """(configuration, number of records) of an export buffer: header checks only, no GPU needed."""
    lib = _lib.load()
    buf = _buffer(data)
    cfg, n = _lib.SameConfig(), C.c_uint32()
    rc = lib.same_state_info(buf.ctypes.data if buf.size else None, buf.size, C.byref(cfg), C.byref(n))
    if rc != 0:
        raise SameEngineError(rc, lib.same_last_error().decode())
    return cfg, n.value


# ---------------------------------------------------------------------------------------------------------------------
# One batch over several GPUs of a box, inside one process (same_multi_* in include/same_engine.h)
# ---------------------------------------------------------------------------------------------------------------------
class SameMultiReceiver:
    """n_streams receivers sharded contiguously over `devices`: one engine + one host thread per device inside the
    native library, no collective (streams are independent).  Events carry global stream ids."""

    def __init__(self, cfg, n_streams: int, devices: Sequence[int]):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self._lib.same_multi_create(C.byref(cfg), devs, len(devices), int(n_streams), C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            raise SameEngineError(rc, self._lib.same_multi_last_error(None).decode())
        self.n_streams = int(n_streams)
        self.devices = [int(d) for d in devices]

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.same_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise SameEngineError(rc, self._lib.same_multi_last_error(self._h).decode())

    def shards(self):
        """[(device, first_stream, n_streams)] per shard."""
        out = []
        for i in range(self._lib.same_multi_num_shards(self._h)):
            d, f, n = C.c_int(), C.c_uint32(), C.c_uint32()
            self._lib.same_multi_shard_info(self._h, i, C.byref(d), C.byref(f), C.byref(n))
            out.append((d.value, f.value, n.value))
        return out

    def set_option(self, key: str, value: int):
        for i in range(len(self.devices)):
            eng = C.c_void_p(self._lib.same_multi_engine(self._h, i))
            rc = self._lib.same_engine_set_option(eng, key.encode(), int(value))
            if rc != 0:
                raise SameEngineError(rc, self._lib.same_engine_last_error(eng).decode())

    def submit(self, chunks):
        flat, offsets, lengths = SameBatchReceiver._pack(chunks)
        if lengths.size != self.n_streams:
            raise ValueError(f"expected {self.n_streams} chunks, got {lengths.size}")
        self._keep = (flat, offsets, lengths)
        self._ck(self._lib.same_multi_submit_s16(self._h, flat.ctypes.data, flat.size, offsets.ctypes.data, lengths.ctypes.data))

    def submit_2d(self, host_ptr: int, row_stride: int, col_start: int, n_cols: int):
        self._ck(self._lib.same_multi_submit_s16_2d(self._h, C.c_void_p(host_ptr), int(row_stride), int(col_start), int(n_cols)))

    def submit_zeros(self, lengths):
        lengths = np.ascontiguousarray(np.broadcast_to(np.asarray(lengths, dtype=np.uint32), (self.n_streams,)))
        self._keep = (lengths,)
        self._ck(self._lib.same_multi_submit_zeros(self._h, lengths.ctypes.data))

    def sync(self):
        self._ck(self._lib.same_multi_sync(self._h))
        self._keep = None

    def reset(self):
        self._ck(self._lib.same_multi_reset(self._h))

    def input_sample_counters(self) -> np.ndarray:
        out = np.zeros(self.n_streams, np.uint64)
        self._ck(self._lib.same_multi_input_sample_counters(self._h, out.ctypes.data))
        return out

    def drain_raw(self):
        nev, npay = C.c_size_t(), C.c_size_t()
        self._ck(self._lib.same_multi_pending(self._h, C.byref(nev), C.byref(npay)))
        evs = np.empty(nev.value, SameBatchReceiver.EVENT_DTYPE)
        pay = np.empty(max(npay.value, 1), np.uint8)
        if nev.value:
            self._ck(self._lib.same_multi_drain_events(self._h, evs.ctypes.data, evs.size, C.byref(nev), pay.ctypes.data,
                                                       pay.size, C.byref(npay)))
        return evs[: nev.value], pay[: npay.value]

    def drain_by_stream(self) -> List[List[SameReceiverEvent]]:
        out: List[List[SameReceiverEvent]] = [[] for _ in range(self.n_streams)]
        for e in SameBatchReceiver.events_from_raw(*self.drain_raw()):
            out[e.stream].append(e)
        return out

    def process(self, chunks) -> List[List[SameReceiverEvent]]:
        self.submit(chunks)
        self.sync()
        return self.drain_by_stream()

    def export_streams(self, ids: Optional[Sequence[int]] = None) -> bytes:
        """SameBatchReceiver.export_streams with global stream ids; records come out in the order of `ids`."""
        return _export(self._lib, self._lib.same_multi_state_bytes, self._lib.same_multi_export_streams, self._h, ids,
                       self.n_streams, self._ck)

    def import_streams(self, data, ids: Optional[Sequence[int]] = None):
        """SameBatchReceiver.import_streams with global stream ids: validated on every shard before any shard changes."""
        _import(self._lib.same_multi_import_streams, self._h, data, ids, self._ck)

    def iter_messages_batched(self, chunks) -> Iterator["tuple[int, Message]"]:
        """== iter_messages (receiver.rs:155-161) for every stream of the whole box: yields (stream, Message)."""
        for evs in self.process(chunks):
            for e in evs:
                m = e.message_ok()
                if m is not None:
                    yield (e.stream, m)


# ---------------------------------------------------------------------------------------------------------------------
# Single-stream facade with the reference's method names
# ---------------------------------------------------------------------------------------------------------------------
class SameReceiver:
    """== SameReceiver (receiver.rs:71-224) backed by a one-stream engine.

    iter_events consumes its input in blocks (the GPU cannot stop mid-block at the first event the way the pull
    iterator does); the events, their order and their input_sample_counter values are identical.
    """

    BLOCK = 1 << 20

    def __init__(self, batch: SameBatchReceiver):
        self._b = batch

    def input_rate(self) -> int:
        return self._b.input_rate()

    def input_sample_counter(self) -> int:
        return int(self._b.input_sample_counters()[0])

    def reset(self):
        self._b.reset()

    def export_state(self) -> bytes:
        """This receiver's complete state as a portable buffer (SameBatchReceiver.export_streams)."""
        return self._b.export_streams()

    def clone(self, device: Optional[int] = None) -> "SameReceiver":
        """== `SameReceiver: Clone` (receiver.rs:70): a new receiver on `device` (default: this one's) in the same
        state; the two share nothing afterwards."""
        return SameReceiver(SameBatchReceiver.from_state(self.export_state(), self._b.device if device is None else device))

    def _blocks(self, source) -> Iterator[np.ndarray]:
        """int16 arrays (and iterables of Python ints) go in as s16 PCM — what samedec feeds (`sa as f32`, app.rs:112);
        anything else is the reference's own f32 item type and goes in as f32, whatever its scale."""
        if isinstance(source, np.ndarray):
            a = source.reshape(-1)
            if a.dtype != np.int16:
                a = a.astype(np.float32, copy=False)
            for i in range(0, a.size, self.BLOCK):
                yield a[i:i + self.BLOCK]
            return
        buf, is_int = [], True
        for v in source:
            is_int = is_int and isinstance(v, (int, np.integer)) and -32768 <= v <= 32767
            buf.append(v)
            if len(buf) >= self.BLOCK:
                yield np.asarray(buf, dtype=np.int16 if is_int else np.float32)
                buf, is_int = [], True
        if buf:
            yield np.asarray(buf, dtype=np.int16 if is_int else np.float32)

    def iter_events(self, source: Iterable) -> Iterator[SameReceiverEvent]:   # receiver.rs:119-130
        for blk in self._blocks(source):
            if blk.dtype == np.int16:
                yield from self._b.process([blk])[0]
            else:
                yield from self._b.process_f32([blk])[0]

    def iter_messages(self, source: Iterable) -> Iterator[Message]:           # receiver.rs:155-161
        for e in self.iter_events(source):
            m = e.message_ok()
            if m is not None:
                yield m

    def flush(self) -> Optional[Message]:                                     # receiver.rs:216-224
        """Four seconds of zeros; returns the first Message and stops consuming AT that sample, as the reference does."""
        nflush = self.input_rate() * 4
        snap = self._b.snapshot()
        try:
            start = self.input_sample_counter()
            self._b.submit_zeros([nflush])
            self._b.sync()
            evs = self._b.drain()
            first = next((e for e in evs if e.message_ok() is not None), None)
            if first is None:
                return None
            # rewind and consume exactly up to the sample that produced the message
            self._b.restore(snap)
            self._b.submit_zeros([first.sample - start])
            self._b.sync()
            self._b.drain()
            return first.message_ok()
        finally:
            self._b.free_snapshot(snap)

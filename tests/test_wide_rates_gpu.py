"""GPU parity tests of the wide-geometry receiver (same_rx_wide_kernel): input rates of 88.2-192 kHz (matched filters of
169-368 taps, up to the 512-tap limit) and DC blockers longer than 64 samples, decoded at the source rate.

Every case compares the events (kind, input_sample_counter, symbol_count, bytes, parity and voting counts) with the CPU
oracle, and the soft-symbol trace bit for bit where it is traced, and asserts that at least one burst was decoded."""
import ctypes as C
import os

import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle
from oracle.pyoracle import OracleConfig, decode_batch_events
from sameold_b200 import _lib, synth

pytestmark = pytest.mark.gpu

EV_BURST, EV_SOM, EV_EOM = 3, 18, 19
ERR_INVALID_ARG, ERR_INVALID_CONFIG = 1, 2


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def builder(rate, samedec=True):
    return sb.SameReceiverBuilder.samedec(rate) if samedec else sb.SameReceiverBuilder.new(rate)


def ocfg(b) -> OracleConfig:
    c, o = b.config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    return o


def oracle(b, x, f32=False):
    o = Oracle(ocfg(b))
    o.enable_trace()
    (o.process_f32 if f32 else o.process_s16)(x)
    return o


def keys(evs):
    return [e.key() for e in evs]


def early_plan(stream_id, rate, seconds, bursts=6, lead=0.3):
    """plan_stream's signal with its first burst `lead` s in, so that a short stream still holds a header; at most
    `bursts` bursts, each complete within `seconds`"""
    p = synth.plan_stream(stream_id, rate, 120.0)
    shift = p.burst_starts[0] - lead * rate
    sym = rate / 520.83
    keep = [(s - shift, b) for s, b in zip(p.burst_starts[:bursts], p.burst_payloads[:bursts])
            if s - shift + len(b) * 8 * sym < seconds * rate]
    return synth.StreamPlan(p.header, [k[0] for k in keep], [k[1] for k in keep], p.freq_offset_hz, p.seed)


def render(stream_id, rate, seconds, **kw):
    return synth.render_numpy(early_plan(stream_id, rate, seconds, **kw), int(seconds * rate), rate)


def check_streams(b, xs, got, rx, what, f32=False, trace=True):
    """events (and the soft trace) of every stream equal to the oracle's; returns the number of bursts decoded"""
    n_bursts = 0
    for s, x in enumerate(xs):
        o = oracle(b, x, f32)
        assert keys(got[s]) == keys(o.events()), f"{what}, stream {s}: events differ from the oracle"
        if trace:
            assert rx.read_soft_trace(s).tobytes() == o.soft_trace().tobytes(), f"{what}, stream {s}: soft trace differs"
        n_bursts += sum(e.kind == EV_BURST for e in got[s])
    return n_bursts


def max_rate_for_taps(ntaps):
    """the largest input rate whose matched filter has at most `ntaps` taps, in the engine's f32 arithmetic"""
    f = lambda r: int(np.floor(np.float32(r) / np.float32(520.83)))
    r = int((ntaps + 1) * 520.83) + 2
    while f(r) > ntaps:
        r -= 1
    while f(r + 1) <= ntaps:
        r += 1
    return r


# ---------------------------------------------------------------------------------------------------------------------
# 1. wide rates, samedec and library-default configurations: a ragged batch plus a noise-only stream, one submit
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("samedec", [True, False], ids=["samedec", "default"])
@pytest.mark.parametrize("rate", [88200, 96000, 176400, 192000])
def test_wide_rates_ragged_batch(rate, samedec):
    _torch()
    b = builder(rate, samedec)
    xs = [render(700 + i, rate, 9.0 + 1.3 * i)[: int((9.0 + 1.3 * i) * rate) - 17 * i] for i in range(3)]
    xs.append(synth.render_numpy(synth.StreamPlan("", [], [], 0.0, 4711), int(6.5 * rate) + 3, rate))   # noise only
    rx = b.build_batch(len(xs))
    assert rx.get_option("kernel_selected") == 1
    assert rx.get_option("resident_blocks_per_sm") >= (2 if rate > 150000 else 4)   # rings sized to the geometry
    assert rx.derived()["ntaps"] == int(np.floor(np.float32(rate) / np.float32(520.83)))
    rx.enable_soft_trace(1 << 16)
    got = rx.process(xs)
    assert not got[-1] or all(e.kind not in (EV_BURST, EV_SOM) for e in got[-1])
    assert check_streams(b, xs, got, rx, f"{rate} Hz") > 0


# ---------------------------------------------------------------------------------------------------------------------
# 2. random chunks of 1..50 000 samples, and odd-width 2-D column slices from pinned memory
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [96000, 192000])
def test_wide_random_chunks(rate):
    _torch()
    b = builder(rate)
    xs = [render(720 + i, rate, 10.0) for i in range(3)]
    n = len(xs[0])
    rng = np.random.default_rng(rate)
    cuts = []
    while sum(cuts) < n:
        cuts.append(1 if rng.random() < 0.1 else int(rng.integers(1, 50001)))
    rx = b.build_batch(len(xs))
    rx.enable_soft_trace(1 << 16)
    got, pos = [[] for _ in xs], 0
    for m in cuts:
        for s, e in enumerate(rx.process([x[pos:pos + m] for x in xs])):
            got[s].extend(e)
        pos += m
    assert check_streams(b, xs, got, rx, f"{rate} Hz random chunks") > 0

    lib = _lib.load()
    stride = n + 3
    hptr = lib.same_host_alloc(len(xs) * stride * 2)
    assert hptr
    try:
        host = np.ctypeslib.as_array(C.cast(hptr, C.POINTER(C.c_int16)), shape=(len(xs), stride))
        for s, x in enumerate(xs):
            host[s, :n] = x
        rx = b.build_batch(len(xs))
        got2, col = [[] for _ in xs], 0
        for width in (1, 7, 55125, 33333, 96001, n):
            w = min(width, n - col)
            if w <= 0:
                break
            rx.submit_2d(hptr, stride, col, w)
            col += w
            rx.sync()
            for s, e in enumerate(rx.drain_by_stream()):
                got2[s].extend(e)
        assert col == n
        for s in range(len(xs)):
            assert keys(got2[s]) == keys(got[s]), f"{rate} Hz 2-D odd chunks, stream {s}"
    finally:
        lib.same_host_free(hptr)


# ---------------------------------------------------------------------------------------------------------------------
# 3. f32 ingest at 96 kHz: normalised samples, library-default AGC limits
# ---------------------------------------------------------------------------------------------------------------------
def test_wide_f32_normalised_96k():
    _torch()
    b = builder(96000, samedec=False)
    xs = [(render(740 + i, 96000, 10.0).astype(np.float32) / np.float32(32768.0)) for i in range(3)]
    rx = b.build_batch(len(xs))
    rx.enable_soft_trace(1 << 16)
    got = rx.process_f32(xs)
    assert check_streams(b, xs, got, rx, "96 kHz f32", f32=True) > 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. DC blockers longer than 64 samples at ordinary rates
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate,length,dc_len", [(22050, 2.0, 84), (48000, 1.0, 92), (192000, 1.0, 368)])
def test_long_dc_blocker(rate, length, dc_len):
    _torch()
    b = builder(rate).with_dc_blocker_length(length)
    xs = [render(760 + i, rate, 9.0) for i in range(2)]
    xs[1] = np.clip(xs[1].astype(np.int32) + 3000, -32768, 32767).astype(np.int16)   # a DC offset to remove
    rx = b.build_batch(len(xs))
    assert rx.derived()["dc_len"] == dc_len
    assert rx.get_option("kernel_selected") == 1
    rx.enable_soft_trace(1 << 16)
    got, pos = [[] for _ in xs], 0
    for m in (dc_len - 1, 1, 5, 100003, len(xs[0])):   # chunks shorter and longer than the window
        for s, e in enumerate(rx.process([x[pos:pos + m] for x in xs])):
            got[s].extend(e)
        pos += m
    assert check_streams(b, xs, got, rx, f"{rate} Hz DC length {dc_len}") > 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. the single-stream facade at 96 kHz: flush() and the forced EOM after 135 s
# ---------------------------------------------------------------------------------------------------------------------
def test_single_stream_facade_96k():
    _torch()
    rate = 96000
    rec = render(780, rate, 9.0, bursts=3)            # header bursts only: the message is pending at EOF
    rx = sb.SameReceiverBuilder.samedec(rate).build()
    assert list(rx.iter_messages(rec)) == []
    m = rx.flush()
    assert m is not None and m.is_start
    o = Oracle(ocfg(sb.SameReceiverBuilder.samedec(rate)))
    o.process_s16(rec)
    o.flush_samedec()
    som = [e for e in o.events() if e.kind == EV_SOM][0]
    assert rx.input_sample_counter() == som.sample
    assert str(m) == bytes(som.data).decode("ascii")
    # 135 s of silence later both force an EndOfMessage (receiver.rs:300-309), at the same sample
    o2 = Oracle(ocfg(sb.SameReceiverBuilder.samedec(rate)))
    o2.process_s16(rec)
    o2.process_zeros(som.sample - len(rec))          # where flush() stopped
    n0 = len(o2.events())
    o2.process_zeros(136 * rate)
    want = o2.events()[n0:]
    got = list(rx.iter_events(np.zeros(136 * rate, np.int16)))
    assert keys(got) == keys(want)
    eom = [e for e in got if e.message_ok() is not None]
    assert [str(e.message_ok()) for e in eom] == ["NNNN"] and eom[0].kind == EV_EOM


# ---------------------------------------------------------------------------------------------------------------------
# 6. limits: 512 taps and DC length 512 accepted, one more refused with the limit named
# ---------------------------------------------------------------------------------------------------------------------
def test_limits():
    _torch()
    top = max_rate_for_taps(512)
    b = builder(top)
    x = [render(800, top, 8.0, bursts=2)]
    rx = b.build_batch(1)
    assert rx.derived()["ntaps"] == 512
    rx.enable_soft_trace(1 << 16)
    got = rx.process(x)
    assert check_streams(b, x, got, rx, f"{top} Hz (512 taps)") > 0

    with pytest.raises(sb.SameEngineError) as ei:
        builder(top + 1).build_batch(1)
    assert ei.value.code == ERR_INVALID_CONFIG
    assert "512" in str(ei.value) and str(top) in str(ei.value)

    sps = np.float32(192000) / np.float32(520.83)
    for want, ok in ((512, True), (513, False)):
        length = float(np.float32(want + 0.5) / sps)
        assert int(np.float32(length) * sps) == want
        bl = builder(192000).with_dc_blocker_length(length)
        if ok:
            assert bl.build_batch(1).derived()["dc_len"] == 512
        else:
            with pytest.raises(sb.SameEngineError) as ei:
                bl.build_batch(1)
            assert ei.value.code == ERR_INVALID_CONFIG and "512" in str(ei.value)


# ---------------------------------------------------------------------------------------------------------------------
# 7. portable state at 192 kHz: export mid-burst, continue in a fresh engine and in a same_multi shard
# ---------------------------------------------------------------------------------------------------------------------
def test_state_192k_mid_burst():
    _torch()
    rate, ns = 192000, 4
    b = builder(rate)
    xs = [render(820 + i, rate, 10.0) for i in range(ns)]
    cut = int(1.1 * rate)                              # inside every stream's first burst (0.3 s .. ~1.5 s)

    whole = b.build_batch(ns).process(xs)
    rx = b.build_batch(ns)
    first = rx.process([x[:cut] for x in xs])
    blob = rx.export_streams()
    cfg, n = sb.state_info(blob)
    assert n == ns and cfg.input_rate == rate and cfg.agc_gain_max == b.config().agc_gain_max
    hdr = 164 + 16 * 368 + 12
    assert int.from_bytes(blob[12:16], "little") == hdr
    rec = int.from_bytes(blob[32:36], "little")
    assert len(blob) == hdr + ns * rec

    fresh = sb.SameBatchReceiver.from_state(blob)
    multi = b.build_multi(ns, [0, 0])
    multi.import_streams(blob)
    rest = [x[cut:] for x in xs]
    ref_after = rx.process(rest)
    for name, r in (("fresh engine", fresh), ("same_multi", multi)):
        after = r.process(rest)
        for s in range(ns):
            assert keys(first[s] + after[s]) == keys(whole[s]), f"{name}, stream {s}"
            assert keys(after[s]) == keys(ref_after[s])
        assert r.export_streams() == rx.export_streams(), name
    assert sum(e.kind == EV_BURST for w in whole for e in w) > 0
    assert any(e.sample > cut and e.kind == EV_BURST for w in whole for e in w)

    with pytest.raises(sb.SameEngineError) as ei:
        builder(96000).build_batch(ns).import_streams(blob)
    assert ei.value.code == ERR_INVALID_CONFIG


# ---------------------------------------------------------------------------------------------------------------------
# 8. one batch larger than the wide kernel's resident capacity at 192 kHz (2 warps of 32 streams per SM)
# ---------------------------------------------------------------------------------------------------------------------
def test_batch_beyond_resident_capacity_192k():
    torch = _torch()
    rate, secs = 192000, 3.0
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ns = (2 * sms + 24) * 32                           # more 32-stream blocks than can be resident at once
    n = int(secs * rate)
    stride = (n + 7) // 8 * 8
    buf = torch.empty((ns, stride), dtype=torch.int16, device="cuda")
    plans = [early_plan(900 + i, rate, secs, bursts=2) for i in range(ns)]
    synth.DeviceCorpus(plans, rate).generate(buf.data_ptr(), stride, n)
    torch.cuda.synchronize()
    b = builder(rate)
    rx = b.build_batch(ns)
    rx.set_event_capacity(ns * 16, ns * 2048)
    offsets = np.arange(ns, dtype=np.uint64) * stride
    rx.submit_device(buf.data_ptr(), ns * stride, offsets, np.full(ns, n, np.uint32))
    rx.sync()
    got = rx.drain_by_stream()
    pick = np.arange(0, ns, 64)
    host = buf[torch.as_tensor(pick, device="cuda"), :n].cpu().numpy()
    ev, pay, _ = decode_batch_events(ocfg(b), host, os.cpu_count() or 1)
    n_bursts = 0
    for j, s in enumerate(pick):
        want = ev[ev["stream"] == j]
        g = got[s]
        assert len(g) == len(want), f"stream {s}: {len(g)} events, the oracle {len(want)}"
        for e, w in zip(g, want):
            data = bytes(pay[w["data_offset"]:w["data_offset"] + w["data_len"]])
            assert (e.kind, e.err, e.sample, e.symbol_count, e.data, e.parity_errors, e.voting_bytes) == \
                (w["kind"], w["err"], w["sample"], w["symbol_count"], data, w["parity_errors"], w["voting_bytes"]), f"stream {s}"
        n_bursts += sum(e.kind == EV_BURST for e in g)
    assert n_bursts > 0

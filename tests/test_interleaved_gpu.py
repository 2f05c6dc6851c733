"""Interleaved multi-channel PCM (same_engine_submit_interleaved / _device, same_multi_submit_interleaved): s16, s24,
s32 and f32 frames deinterleaved on the GPU, one channel per stream.

Every case compares against planar submits of the same channels on a second engine: s16 through `submit`, s24 / s32 /
f32 through `submit_f32` of `x.astype(np.float32)` (the reference's `sa as f32`).  Events, soft-symbol trace and the
exported resident state must be equal after every submit, and every case must decode at least one burst.  A subset is
also compared with the CPU oracle."""
import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle
from oracle.pyoracle import OracleConfig
from sameold_b200 import synth
from sameold_b200.receiver import CHANNEL_SKIP

pytestmark = pytest.mark.gpu

EV_BURST = 3
FORMATS = ["s16", "s24", "s32", "f32"]
SECONDS = 8.0


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def channel_s16(c, rate, n):
    """channel c: a seeded synth stream whose first burst starts at 0.5 + 0.15 c s, over corpus noise; channel 1 is
    silent and channel 2 at full scale (clipped) when there are that many"""
    if c == 1:
        return np.zeros(n, np.int16)
    p = synth.plan_stream(700 + c, rate, 120.0)
    shift = p.burst_starts[0] - (0.5 + 0.15 * c) * rate
    plan = synth.StreamPlan(p.header, [s - shift for s in p.burst_starts], p.burst_payloads, p.freq_offset_hz, p.seed)
    return synth.render_numpy(plan, n, rate, amplitude=40000.0 if c == 2 else synth.AMPLITUDE)


_CACHE = {}


def channels(rate, n_channels):
    n = int(SECONDS * rate)
    key = rate
    if key not in _CACHE or _CACHE[key].shape[1] < n_channels:
        _CACHE[key] = np.stack([channel_s16(c, rate, n) for c in range(33)], axis=1)
    return _CACHE[key][:, :n_channels]


def as_format(x16, fmt, seed=0):
    """int16 frames [n, C] -> frames of `fmt` carrying the same signal, with low bits that exercise the conversion:
    (2-D array, or bytes for s24)"""
    rng = np.random.default_rng(seed)
    x = x16.astype(np.int64)
    if fmt == "s16":
        return x16.copy()
    if fmt == "s24":
        v = x * 256 + rng.integers(0, 256, x.shape)
        return pack_s24(v)
    if fmt == "s32":
        return (x * 65536 + rng.integers(0, 65536, x.shape)).astype(np.int32)
    # samedec's AGC limits ([1/32767, 1/200]) want s16 scale; the fractions keep the DC state off the integers
    return (x16.astype(np.float32) + rng.uniform(-0.5, 0.5, x.shape).astype(np.float32)).astype(np.float32)


def pack_s24(v):
    u = (np.asarray(v, np.int64) & 0xFFFFFF).astype(np.uint32)
    b = np.stack([u & 0xFF, (u >> 8) & 0xFF, (u >> 16) & 0xFF], axis=-1).astype(np.uint8)
    return b.reshape(-1).tobytes()


def values(frames, fmt, n_channels):
    """the samples `frames` carries, [n, C], as int16 (s16) or as their exact integer / float value"""
    if fmt == "s24":
        b = np.frombuffer(frames, np.uint8).reshape(-1, n_channels, 3).astype(np.int32)
        v = b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)
        return np.where(v >= 1 << 23, v - (1 << 24), v)
    return frames


def submit_il(rx, frames, fmt, n_channels, cmap=None):
    if fmt == "s24":
        rx.submit_interleaved(frames, cmap, fmt="s24", n_channels=n_channels)
    else:
        rx.submit_interleaved(frames, cmap)


def submit_planar(rx, vals, fmt, cmap, n_streams):
    """the reference arm: stream cmap[c] <- column c, planar"""
    n = vals.shape[0]
    rows = [None] * n_streams
    for c in range(vals.shape[1]):
        s = c if cmap is None else cmap[c]
        if s is None or s < 0 or s == CHANNEL_SKIP:
            continue
        rows[s] = vals[:, c]
    if fmt == "s16":
        rx.submit([np.zeros(0, np.int16) if r is None else np.ascontiguousarray(r, np.int16) for r in rows])
    else:
        rx.submit_f32([np.zeros(0, np.float32) if r is None else np.asarray(r).astype(np.float32) for r in rows])


def state_only(blob):
    """the records of an export without their flags word and CRC: the flags carry the engine-wide f32 bit"""
    hdr = int.from_bytes(blob[12:16], "little")
    n, rec = int.from_bytes(blob[16:20], "little"), int.from_bytes(blob[32:36], "little")
    recs = np.frombuffer(blob[hdr:hdr + n * rec], np.uint8).reshape(n, rec)
    return np.concatenate([recs[:, :4], recs[:, 8:rec - 4]], axis=1).tobytes()


def engine(rate, n_streams, trace=True):
    rx = sb.SameReceiverBuilder.samedec(rate).build_batch(n_streams)
    if trace:
        rx.enable_soft_trace(1 << 16)
    return rx


def keys(evs):
    return [(e.stream,) + e.key() for e in evs]


def assert_same(a, b, what, n_streams, trace=True):
    """events, soft trace and exported state of two engines (after sync)"""
    ea, eb = a.drain(), b.drain()
    assert keys(ea) == keys(eb), f"{what}: events differ"
    if trace:
        for s in range(n_streams):
            assert a.read_soft_trace(s).tobytes() == b.read_soft_trace(s).tobytes(), f"{what}: soft trace of stream {s}"
    assert a.export_streams() == b.export_streams(), f"{what}: exported state differs"
    return ea


def bursts(evs):
    return sum(e.kind == EV_BURST for e in evs)


def ocfg(rate):
    c, o = sb.SameReceiverBuilder.samedec(rate).config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    return o


# ---- 1. formats x channel counts x rates ----
@pytest.mark.parametrize("rate", [22050, 48000, 96000])
@pytest.mark.parametrize("n_channels", [1, 2, 3, 8, 33])
@pytest.mark.parametrize("fmt", FORMATS)
def test_formats_and_rates(fmt, n_channels, rate):
    x16 = channels(rate, n_channels)
    frames = as_format(x16, fmt, seed=n_channels)
    vals = values(frames, fmt, n_channels)
    a, b = engine(rate, n_channels), engine(rate, n_channels)
    half = x16.shape[0] // 2 + 3   # two submits, the first not a multiple of 8 frames
    fb = {"s24": 3}.get(fmt, 0) * n_channels
    for lo, hi in ((0, half), (half, x16.shape[0])):
        part = frames[lo * fb:hi * fb] if fmt == "s24" else frames[lo:hi]
        submit_il(a, part, fmt, n_channels)
        submit_planar(b, vals[lo:hi], fmt, None, n_channels)
        a.sync(); b.sync()
        evs = assert_same(a, b, f"{fmt} C={n_channels} {rate} Hz", n_channels)
        if lo == 0:
            first = evs
    assert bursts(first + evs) >= 1
    if fmt == "s16":
        assert a.get_option("kernel_selected") == b.get_option("kernel_selected")
    else:
        assert a.get_option("kernel_selected") == 1
    # the oracle for a subset: one channel of each case with two or three channels
    if n_channels in (2, 3):
        c = n_channels - 1 if n_channels == 2 else 0
        o = Oracle(ocfg(rate))
        o.enable_trace()
        if fmt == "s16":
            o.process_s16(np.ascontiguousarray(vals[:, c]))
        else:
            o.process_f32(np.ascontiguousarray(vals[:, c]).astype(np.float32))
        a3 = engine(rate, n_channels)
        evs = a3.process_interleaved(*((frames, None, "s24", n_channels) if fmt == "s24" else (frames,)))
        assert [e.key() for e in evs[c]] == [e.key() for e in o.events()], f"{fmt} C={n_channels} {rate}: oracle"
        assert a3.read_soft_trace(c).tobytes() == o.soft_trace().tobytes()


# ---- 2. chunking ----
@pytest.mark.parametrize("fmt", FORMATS)
def test_random_chunks_from_odd_host_addresses(fmt):
    rate, C = 22050, 3
    x16 = channels(rate, C)
    frames = as_format(x16, fmt, seed=5)
    raw = frames if fmt == "s24" else frames.tobytes()
    fb = len(raw) // x16.shape[0]
    odd = np.zeros(len(raw) + 1, np.uint8)
    odd[1:] = np.frombuffer(raw, np.uint8)
    assert odd[1:].ctypes.data % 2 == 1
    whole, chunked = engine(rate, C), engine(rate, C)
    whole.submit_interleaved(raw, None, fmt=fmt, n_channels=C)
    whole.sync()
    rng = np.random.default_rng(11)
    pos, k, evs = 0, 0, []
    while pos < x16.shape[0]:
        m = int(rng.integers(1, 50001))
        chunked.submit_interleaved(odd[1 + pos * fb:1 + min(pos + m, x16.shape[0]) * fb], None, fmt=fmt, n_channels=C)
        pos = min(pos + m, x16.shape[0])
        k += 1
        if k % 2 == 0:   # two submits in flight between syncs
            chunked.sync()
    chunked.sync()
    evs = assert_same(chunked, whole, f"{fmt} chunked", C)
    assert k > 3 and bursts(evs) >= 1


# ---- 3. channel maps and rejections ----
@pytest.mark.parametrize("fmt", ["s16", "s24"])
def test_channel_maps(fmt):
    rate = 22050
    x16 = channels(rate, 4)
    frames = as_format(x16, fmt, seed=3)
    vals = values(frames, fmt, 4)
    for cmap in ([3, 0, 5, 1], [2, CHANNEL_SKIP, 0, CHANNEL_SKIP], [5, None, -1, 4]):
        a, b = engine(rate, 6), engine(rate, 6)
        fed = {s for s in cmap if s is not None and s >= 0 and s != CHANNEL_SKIP}
        unfed = [s for s in range(6) if s not in fed]
        before = a.export_streams(unfed)
        submit_il(a, frames, fmt, 4, cmap)
        submit_planar(b, vals, fmt, [CHANNEL_SKIP if s is None or s < 0 else s for s in cmap], 6)
        a.sync(); b.sync()
        assert state_only(a.export_streams(unfed)) == state_only(before), f"{cmap}: unfed streams changed"
        evs = assert_same(a, b, f"{fmt} map {cmap}", 6)
        assert bursts(evs) >= 1
    # stereo, one channel kept, one-stream engine
    a, b = engine(rate, 1), engine(rate, 1)
    st = pack_s24(vals[:, 2:4]) if fmt == "s24" else frames[:, 2:4]
    submit_il(a, st, fmt, 2, [CHANNEL_SKIP, 0])
    submit_planar(b, vals[:, 2:4], fmt, [CHANNEL_SKIP, 0], 1)
    a.sync(); b.sync()
    assert bursts(assert_same(a, b, "stereo, right channel kept", 1)) >= 1


def test_rejections_change_nothing():
    rate, C = 22050, 4
    x16 = channels(rate, C)
    rx = engine(rate, 4, trace=False)
    rx.process_interleaved(x16[:20000])
    state = rx.export_streams()
    lib = rx._lib
    cases = [
        (x16.ctypes.data, 7, 4, 100, None, "format"),
        (x16.ctypes.data, 0, 0, 100, None, "n_channels"),
        (x16.ctypes.data, 0, 4, (1 << 30) + 1, None, "2^30"),
        (x16.ctypes.data, 0, 4, 100, [0, 1, 9, 2], "channel 2"),
        (x16.ctypes.data, 0, 4, 100, [0, 1, 2, 1], "channel 3"),
        (None, 0, 4, 100, None, "null"),
        (x16.ctypes.data, 0, 5, 100, None, "channel 4"),
    ]
    for ptr, fmt, nc, nf, cmap, word in cases:
        m = None if cmap is None else np.array(cmap, np.uint32)
        for fn in (lib.same_engine_submit_interleaved, lib.same_engine_submit_interleaved_device):
            rc = fn(rx.handle, ptr, fmt, nc, nf, None if m is None else m.ctypes.data)
            assert rc == 1, (word, rc)
            assert word in lib.same_engine_last_error(rx.handle).decode(), lib.same_engine_last_error(rx.handle)
    rx.sync()
    assert rx.export_streams() == state
    with pytest.raises(sb.SameEngineError) as ei:
        rx.submit_interleaved(x16, [0, 0, 1, 2])
    assert "channel 1" in str(ei.value)
    assert rx.export_streams() == state
    assert rx.get_option("kernel_selected") != 1   # not put on the f32 path by a refused submit


# ---- 4. value edges ----
EDGES = {
    "s16": [-32768, 32767, -32768, 32767],
    "s24": [-8388608, 8388607, -8388608, 8388607],
    "s32": [-(1 << 31), (1 << 31) - 1, (1 << 24) + 1, (1 << 24) + 3, -(1 << 24) - 1, -(1 << 24) - 3, (1 << 25) + 2],
    "f32": [0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, -5e-40, 1e30, -1e30],
}


@pytest.mark.parametrize("fmt", FORMATS)
def test_value_edges(fmt):
    rate = 22050
    x16 = channels(rate, 2)
    frames = as_format(x16, fmt, seed=9)
    vals = np.array(values(frames, fmt, 2), copy=True)
    edge = np.array(EDGES[fmt], dtype={"s16": np.int16, "s24": np.int64, "s32": np.int32, "f32": np.float32}[fmt])
    reps = np.tile(edge, 64)
    vals[1000:1000 + reps.size, 1] = reps   # channel 1: silent, then the edge values
    if fmt == "f32":
        assert np.signbit(vals[1001, 1]) and vals[1002, 1] != 0
    frames = pack_s24(vals) if fmt == "s24" else vals
    a, b = engine(rate, 2), engine(rate, 2)
    submit_il(a, frames, fmt, 2)
    submit_planar(b, vals, fmt, None, 2)
    a.sync(); b.sync()
    assert bursts(assert_same(a, b, f"{fmt} edges", 2)) >= 1
    if fmt == "s32":   # round to nearest even, as numpy's int32 -> float32
        assert np.float32(np.int32((1 << 24) + 1)) == np.float32(1 << 24)
        assert np.float32(np.int32((1 << 24) + 3)) == np.float32((1 << 24) + 4)


# ---- 5. path selection ----
def test_path_selection():
    rate, C = 22050, 2
    x16 = channels(rate, C)
    for fmt in FORMATS:
        a = engine(rate, 64, trace=False)
        planar = engine(rate, 64, trace=False)
        frames = as_format(x16, fmt)
        submit_il(a, frames, fmt, C)
        a.sync()
        if fmt == "s16":
            planar.submit([x16[:, 0], x16[:, 1]] + [None] * 62)
            planar.sync()
            assert a.get_option("kernel_selected") == planar.get_option("kernel_selected") != 1
        else:
            assert a.get_option("kernel_selected") == 1, fmt
            a.reset()
            assert a.get_option("kernel_selected") == planar.get_option("kernel_selected") != 1


@pytest.mark.parametrize("rate", [22050, 48000])
def test_long_path_from_one_channel_of_stereo(rate):
    n = int(12 * rate)
    assert n >= 65536
    mono = channel_s16(0, rate, n)
    stereo = np.stack([mono, channel_s16(3, rate, n)], axis=1)
    runs = []
    for long_stream in (1, 0):
        rx = engine(rate, 1)
        rx.set_option("long_stream", long_stream)
        got = []
        for lo in range(0, n, 100000):
            got += rx.process_interleaved(stereo[lo:lo + 100000], [0, CHANNEL_SKIP])[0]
        runs.append((rx, got, rx.export_streams(), rx.read_soft_trace(0).tobytes()))
    (rx1, g1, s1, t1), (rx0, g0, s0, t0) = runs
    assert rx1.get_option("long_stream_passes") >= 1 and rx0.get_option("long_stream_passes") == 0
    assert [e.key() for e in g1] == [e.key() for e in g0] and s1 == s0 and t1 == t0
    assert bursts(g1) >= 1


# ---- 6. device variant ----
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("offset", [0, 1])
def test_device_frames(fmt, offset):
    torch = _torch()
    rate, C = 22050, 3
    x16 = channels(rate, C)
    frames = as_format(x16, fmt, seed=offset)
    raw = frames if fmt == "s24" else frames.tobytes()
    d = torch.zeros(len(raw) + 16, dtype=torch.uint8, device="cuda")
    d[offset:offset + len(raw)] = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    a, b = engine(rate, C), engine(rate, C)
    n = x16.shape[0]
    a.submit_interleaved_device(d.data_ptr() + offset, fmt, C, n, [2, 0, 1])
    b.submit_interleaved(raw, [2, 0, 1], fmt=fmt, n_channels=C)
    a.sync(); b.sync()
    assert bursts(assert_same(a, b, f"device {fmt} +{offset}", C)) >= 1
    del d


# ---- 7. several devices ----
@pytest.mark.parametrize("devices", [[0, 0], [0, 1]])
def test_multi(devices):
    torch = _torch()
    if max(devices) >= torch.cuda.device_count():
        pytest.skip("needs two GPUs")
    rate, C, n_streams = 22050, 8, 6
    x16 = channels(rate, C)
    cmap = [5, CHANNEL_SKIP, 0, 3, 1, CHANNEL_SKIP, 4, 2]
    for fmt in ("s16", "s24"):
        frames = as_format(x16, fmt, seed=2)
        cfg = sb.SameReceiverBuilder.samedec(rate).config()
        m = sb.SameMultiReceiver(cfg, n_streams, devices)
        one = engine(rate, n_streams, trace=False)
        half = x16.shape[0] // 2
        fb = 3 * C if fmt == "s24" else 0
        for lo, hi in ((0, half), (half, x16.shape[0])):
            part = frames[lo * fb:hi * fb] if fmt == "s24" else frames[lo:hi]
            submit_il(m, part, fmt, C, cmap)
            submit_il(one, part, fmt, C, cmap)
            m.sync(); one.sync()
            got = m.drain_by_stream()
            want = one.drain_by_stream()
            assert [[(e.stream,) + e.key() for e in s] for s in got] == [[(e.stream,) + e.key() for e in s] for s in want]
            assert m.export_streams() == one.export_streams()
        m.close()

"""The long-stream path at every geometry the engine accepts (same_long.cu: the general DC front, the AGC and sequential
kernels at any tap count, the wide matched filter; bursts and unverified spans by the generic or wide kernel): one
s16 stream at 11 025, 44 100, 48 000, 96 000 and 192 000 Hz, 22 050 Hz with DC length 84, and the 512-tap / DC-512
top geometry.

Every case compares events and the soft-symbol trace with the CPU oracle, and the exported resident state after every
chunk with long_stream = 0 (the same engine's ordinary kernels), and asserts that the long path ran."""
import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle
from oracle.pyoracle import OracleConfig
from sameold_b200 import synth

pytestmark = pytest.mark.gpu

EV_BURST, EV_SOM, EV_EOM = 3, 18, 19
F_DC_FBSUM = 32


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def ocfg(b) -> OracleConfig:
    c, o = b.config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    return o


def oracle(b, x):
    o = Oracle(ocfg(b))
    o.enable_trace()
    o.process_s16(x)
    return o


def keys(evs):
    return [e.key() for e in evs]


def max_rate_for_taps(ntaps):
    f = lambda r: int(np.floor(np.float32(r) / np.float32(520.83)))
    r = int((ntaps + 1) * 520.83) + 2
    while f(r) > ntaps:
        r -= 1
    while f(r + 1) <= ntaps:
        r += 1
    return r


def event_plan(rate, events, first=1.0, gap=3.0, seed=0):
    """`events` SAME events (3 header + 3 EOM bursts each, from plan_stream) one after another from `first` s on;
    (plan, burst intervals in samples, end of the last burst in samples)"""
    starts, pays, t, header = [], [], first * rate, ""
    for k in range(events):
        p = synth.plan_stream(600 + 7 * seed + k, rate, 120.0)
        header = header or p.header
        shift = p.burst_starts[0] - t
        starts += [s - shift for s in p.burst_starts]
        pays += p.burst_payloads
        t = starts[-1] + len(pays[-1]) * 8 * rate / 520.83 + gap * rate
    spans = [(s, s + len(q) * 8 * rate / 520.83) for s, q in zip(starts, pays)]
    return synth.StreamPlan(header, starts, pays, 1.7, 0x5EED + seed), spans, int(t)


def event_stream(rate, events=2, zeros_s=20.0, seed=0, **kw):
    """events over corpus noise, then `zeros_s` s of exact zeros; (samples, burst intervals)"""
    plan, spans, n = event_plan(rate, events, seed=seed)
    x = synth.render_numpy(plan, n, rate, **kw)
    return np.concatenate([x, np.zeros(int(zeros_s * rate), np.int16)]), spans


def ragged(n, rate, seed, lo=65536, hi=400000):
    rng, out = np.random.default_rng(seed), []
    k = rate / 22050.0
    while sum(out) < n:
        out.append(int(rng.integers(int(lo * k), int(hi * k) + 1)))
    return out


def run(b, x, lens, long_stream, trace=True):
    """one one-stream engine over x in chunks: (events, exported state after every chunk, engine)"""
    rx = b.build_batch(1)
    rx.set_option("long_stream", long_stream)
    if trace:
        rx.enable_soft_trace(1 << 18)
    got, exports, pos = [], [], 0
    for m in lens:
        got.extend(rx.process([x[pos:pos + m]])[0])
        exports.append(rx.export_streams())
        pos += m
    assert pos >= len(x)
    return got, exports, rx


def state_words(blob):
    hdr = int.from_bytes(blob[12:16], "little")
    head = np.frombuffer(blob[:36], "<u4")
    n, n_words, rec = int(head[4]), int(head[5]), int(head[8])
    recs = np.frombuffer(blob[hdr:hdr + n * rec], np.uint8).reshape(n, rec)
    return recs[:, 8:8 + 4 * n_words].copy().view("<u4")


def check_parity(b, x, lens, what, trace=True):
    """long path against the oracle and against long_stream = 0; returns (events, passes, fallback spans, exports)"""
    got, exp, rx = run(b, x, lens, 1, trace)
    ref_got, ref_exp, _ = run(b, x, lens, 0, trace)
    o = oracle(b, x)
    assert keys(got) == keys(o.events()), f"{what}: events differ from the oracle"
    assert keys(ref_got) == keys(got)
    if trace:
        assert rx.read_soft_trace(0).tobytes() == o.soft_trace().tobytes(), f"{what}: soft trace differs"
    for k in range(len(lens)):
        assert exp[k] == ref_exp[k], f"{what}: state differs from long_stream = 0 after chunk {k}"
    assert rx.get_option("kernel_selected") == 1
    return got, rx.get_option("long_stream_passes"), rx.get_option("long_stream_fallback_spans"), exp


# ---------------------------------------------------------------------------------------------------------------------
# 1. every geometry class, whole and in ragged chunks whose boundaries fall inside bursts
# ---------------------------------------------------------------------------------------------------------------------
GEOMETRIES = [(11025, None), (44100, None), (48000, None), (96000, None), (192000, None), (22050, 2.0), ("top", "top")]


@pytest.mark.parametrize("rate,dc", GEOMETRIES, ids=["11k", "44k1", "48k", "96k", "192k", "22k05-dc84", "512-taps-dc512"])
def test_long_path_at_every_geometry(rate, dc):
    _torch()
    if rate == "top":
        rate = max_rate_for_taps(512)
        sps = np.float32(rate) / np.float32(520.83)
        b = sb.SameReceiverBuilder.samedec(rate).with_dc_blocker_length(float(np.float32(512.5) / sps))
    else:
        b = sb.SameReceiverBuilder.samedec(rate)
        if dc is not None:
            b = b.with_dc_blocker_length(dc)
    d = b.build_batch(1).derived()
    if rate > 260000:
        assert d["ntaps"] == 512 and d["dc_len"] == 512
    if dc == 2.0:
        assert d["dc_len"] == 84
    x, spans = event_stream(rate, events=2, seed=rate % 97)
    cuts = ragged(len(x), rate, seed=rate)
    bounds = np.cumsum(cuts)[:-1]
    assert any(s0 < c < s1 for c in bounds for s0, s1 in spans), "a chunk boundary inside a burst"
    for chunking, lens in (("whole", [len(x)]), ("ragged", cuts)):
        got, passes, fb, _ = check_parity(b, x, lens, f"{rate} Hz dc_len {d['dc_len']}, {chunking}")
        assert passes >= 1 and fb >= 1, (chunking, passes, fb)
        assert sum(e.kind == EV_BURST for e in got) >= 6 and any(e.kind == EV_SOM for e in got)


# ---------------------------------------------------------------------------------------------------------------------
# 2. quiet levels at 48 kHz: verification stops and unverified spans
# ---------------------------------------------------------------------------------------------------------------------
def test_long_path_at_quiet_levels_48k():
    _torch()
    rate = 48000
    b = sb.SameReceiverBuilder.samedec(rate)
    noise = lambda sigma, sec, seed: synth.render_numpy(synth.StreamPlan("", [], [], 0.0, seed), int(sec * rate), rate,
                                                        noise_sigma=sigma)
    plan, _, n = event_plan(rate, 3, first=15.0, gap=20.0, seed=3)
    cases = {"noise 500": noise(500.0, 150.0, 11), "noise 3663": noise(3663.0, 120.0, 12),
             "bursts 2000 over 500": synth.render_numpy(plan, n + 10 * rate, rate, amplitude=2000.0, noise_sigma=500.0)}
    for name, x in cases.items():
        for chunking, lens in (("whole", [len(x)]), ("ragged", ragged(len(x), rate, 5, 65536, 3 * 65536))):
            got, passes, spans, _ = check_parity(b, x, lens, f"48 kHz {name}, {chunking}")
            starts = np.cumsum([0] + lens[:-1])
            big = [m for m, s0 in zip(lens, starts) if min(m, len(x) - s0) >= 65536]
            if name == "noise 500":
                assert passes >= 2 * len(big) and spans >= 1, (chunking, passes, spans)
            if name == "noise 3663":
                assert passes == len(big) and spans == 0, (chunking, passes, spans)
            if name.startswith("bursts"):
                assert any(e.kind == EV_SOM for e in got) and spans >= 1


# ---------------------------------------------------------------------------------------------------------------------
# 3. DC stress at 44.1 and 48 kHz: the feedback sum leaves the exact range, the DC words must still match
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [44100, 48000])
def test_long_path_dc_stress(rate):
    _torch()
    b = sb.SameReceiverBuilder.samedec(rate)
    x, _ = event_stream(rate, events=1, zeros_s=2.0, seed=9)
    x = np.clip(x.astype(np.int32) + 20000, -32768, 32767).astype(np.int16)          # +20 000 DC offset
    n = len(x)
    alt = np.tile(np.array([32767, -32768], np.int16), rate)                          # 2 s full-scale alternation
    steps = np.where((np.arange(rate) // 331) % 2 == 0, 32767, -32768).astype(np.int16)   # rail-to-rail steps
    neg = np.full(3 * rate, -20000, np.int16)
    x = np.concatenate([x[: n // 2], alt, steps, neg, x[n // 2:]])
    for chunking, lens in (("whole", [len(x)]), ("ragged", ragged(len(x), rate, 17))):
        got, passes, _, exp = check_parity(b, x, lens, f"{rate} Hz DC stress, {chunking}")
        assert passes >= 1
    fb = np.array([state_words(e)[0, F_DC_FBSUM] for e in exp], np.uint32).view(np.float32)
    assert np.max(np.abs(fb)) > 2 ** 19, "the feedback sum reached beyond the exact range"


# ---------------------------------------------------------------------------------------------------------------------
# 4. mixed submits, a mid-burst record continued with a long chunk, the one-stream facade
# ---------------------------------------------------------------------------------------------------------------------
def test_mixed_submits_and_mid_burst_import_48k():
    _torch()
    rate = 48000
    b = sb.SameReceiverBuilder.samedec(rate)
    x, spans = event_stream(rate, events=2, zeros_s=5.0, seed=21)
    a, c = int(spans[1][0] + 0.4 * rate), int(spans[4][0] + 0.3 * rate)
    engines = []
    for ls in (1, 0):
        rx = b.build_batch(1)
        rx.set_option("long_stream", ls)
        got = rx.process([x[:a]])[0] + rx.process([x[a:a + 5000]])[0]
        rx.submit_zeros([7777])
        rx.sync()
        got += rx.drain()
        got += rx.process([x[a + 5000:]])[0]
        engines.append((got, rx.export_streams(), rx.get_option("long_stream_passes")))
    assert keys(engines[0][0]) == keys(engines[1][0]) and engines[0][1] == engines[1][1]
    assert engines[0][2] >= 2 and engines[1][2] == 0

    # export inside a burst, import into a one-stream engine, continue with one long chunk
    whole = oracle(b, x).events()
    src = b.build_batch(1)
    first = src.process([x[:c]])[0]
    blob = src.export_streams()
    for ls in (1, 0):
        dst = sb.SameBatchReceiver.from_state(blob)
        dst.set_option("long_stream", ls)
        after = dst.process([x[c:]])[0]
        assert keys(first + after) == keys(whole), f"long_stream {ls}"
        if ls:
            assert dst.get_option("long_stream_passes") >= 1 and dst.get_option("long_stream_fallback_spans") >= 1
            blob_long = dst.export_streams()
        else:
            assert dst.export_streams() == blob_long


def test_single_stream_facade_48k():
    _torch()
    rate = 48000
    plan, spans, _ = event_plan(rate, 1, first=2.0)
    plan = synth.StreamPlan(plan.header, plan.burst_starts[:3], plan.burst_payloads[:3], plan.freq_offset_hz, plan.seed)
    # header bursts only, the recording ending 0.2 s after the third: the message is still pending at EOF
    rec = synth.render_numpy(plan, int(spans[2][1] + 0.2 * rate), rate)
    assert len(rec) >= 4 * 65536
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
    # with 30 s of noise after the bursts the assembler's deadline passes inside the recording: the message comes out
    # of iter_messages, as the oracle's does
    tail = np.concatenate([rec, synth.render_numpy(synth.StreamPlan("", [], [], 0.0, 5), 30 * rate, rate)])
    rx = sb.SameReceiverBuilder.samedec(rate).build()
    got = [str(x) for x in rx.iter_messages(tail)]
    o = oracle(sb.SameReceiverBuilder.samedec(rate), tail)
    assert got == [bytes(e.data).decode("ascii") for e in o.events() if e.kind in (EV_SOM, EV_EOM)] and len(got) == 1


# ---------------------------------------------------------------------------------------------------------------------
# 5. the path not taken: after f32 input, with "kernel" forced, on a 2-stream engine
# ---------------------------------------------------------------------------------------------------------------------
def test_long_path_not_taken_48k():
    _torch()
    rate = 48000
    b = sb.SameReceiverBuilder.samedec(rate)
    x, _ = event_stream(rate, events=1, zeros_s=1.0, seed=31)
    want = keys(oracle(b, x).events())
    rx = b.build_batch(1)
    got = rx.process_f32([x[:1000].astype(np.float32)])[0] + rx.process([x[1000:]])[0]
    assert rx.get_option("long_stream_passes") == 0
    assert keys(got) == want
    rx = b.build_batch(1)
    rx.set_option("kernel", 1)
    assert keys(rx.process([x])[0]) == want and rx.get_option("long_stream_passes") == 0
    rx = b.build_batch(2)
    got = rx.process([x, x[: len(x) // 2]])
    assert keys(got[0]) == want and rx.get_option("long_stream_passes") == 0
    rx = b.build_batch(1)                                    # and taken on the same input otherwise
    assert keys(rx.process([x])[0]) == want and rx.get_option("long_stream_passes") >= 1


# ---------------------------------------------------------------------------------------------------------------------
# 6. a 2 h stream at 48 kHz from the device generator, in 10-minute chunks, against the oracle event for event
# ---------------------------------------------------------------------------------------------------------------------
def test_two_hour_stream_48k():
    torch = _torch()
    rate, hours = 48000, 2.0
    n = int(hours * 3600 * rate)
    plan = synth.plan_long_stream(hours, rate)
    buf = torch.empty(((n + 7) // 8 * 8,), dtype=torch.int16, device="cuda")
    synth.DeviceCorpus([plan], rate).generate(buf.data_ptr(), buf.numel(), n)
    torch.cuda.synchronize()
    b = sb.SameReceiverBuilder.samedec(rate)
    rx = b.build_batch(1)
    step, got = 600 * rate, []
    for lo in range(0, n, step):
        k = min(step, n - lo)
        rx.submit_device(buf.data_ptr() + 2 * lo, k, np.zeros(1, np.uint64), np.array([k], np.uint32))
        rx.sync()
        got.extend(rx.drain())
    assert rx.input_sample_counters()[0] == n
    assert rx.get_option("long_stream_passes") >= n // step
    o = Oracle(ocfg(b))
    o.process_s16(buf[:n].cpu().numpy())
    want = o.events()
    assert sum(e.kind in (EV_SOM, EV_EOM) for e in want) >= 2
    assert keys(got) == keys(want)

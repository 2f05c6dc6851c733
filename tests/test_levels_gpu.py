"""GPU parity tests away from the corpus's one operating point (16384-amplitude bursts over sigma 3663 noise at exactly
520.83 Bd): burst levels from barely decodable to overdriven and clipped, noise from none to the corpus level, DC
offsets and steps, the worst-case input of the integer DC blocker, off-rate symbols, f32 input at extreme scales, and
the long-stream path on quiet noise where its speculative AGC hand-overs fail to verify.

Every case compares events and the soft-symbol trace with the CPU oracle, and the resident state (export_streams)
after every chunk with the rate-generic kernel's on the same chunks.  Each case also asserts that it reached the regime
it is for: the AGC gain pinned at either limit, the timing loop's period at its clamp, verification stops of the long
path, roll-backs of the pipelined kernel."""
import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle, load_golden_recording
from oracle.pyoracle import OracleConfig
from sameold_b200 import synth

pytestmark = pytest.mark.gpu

RATE = 22050
BAUD = 520.83
NAMES = ["long_message", "npt", "two_and_two"]
HEADER = synth.PREAMBLE + b"ZCZC-WXR-TOR-029165-029169+0030-1051700-KEAX/NWS-"
EOM = synth.PREAMBLE + b"NNNN"
EV_BURST, EV_SOM, EV_EOM = 3, 18, 19

# state words (sameold_b200/csrc/same_params.h: SameField, and the array layout same_engine.cu builds after the scalars)
F_AGC_GAIN, F_FLAGS, F_PAVG, F_DC_FFSUM, F_DC_FBSUM, F_NUM_SCALARS = 0, 1, 4, 31, 32, 34
HEADER_BYTES, RECORD_WORDS_AT = 2224, 8


# ---------------------------------------------------------------------------------------------------------------------
# Deterministic test-signal renderer (numpy only; tests/test_levels_cpu.py checks it on the CPU)
# ---------------------------------------------------------------------------------------------------------------------
def render(n, bursts=(), sigma=0.0, seed=0, dc=0.0, dc_step=None, rate=RATE, foff=1.5, splice=()):
    """int16 samples [n] of a SAME signal: `bursts` = (start sample, payload bytes, amplitude, baud) AFSK bursts (mark
    2083.3 Hz, space 1562.5 Hz, phase-continuous, LSB first), plus Gaussian noise of `sigma` LSB (Philox, `seed`), plus
    a DC offset `dc` and a step dc_step = (sample, delta) to dc + delta from that sample on; rounded and clipped to
    s16.  `splice` = (sample, int16 array) pieces written over the result afterwards."""
    t = np.arange(n, dtype=np.float64)
    sig = np.zeros(n, np.float64)
    fm, fs = 2083.3 + foff, 1562.5 + foff
    for start, payload, amp, baud in bursts:
        ts = rate / baud
        bits = np.unpackbits(np.frombuffer(payload, np.uint8), bitorder="little").astype(np.int64)
        i0, i1 = int(np.ceil(start)), min(n, int(np.ceil(start + len(bits) * ts)))
        if i1 <= i0:
            continue
        tt = t[i0:i1] - start
        k = np.minimum((tt / ts).astype(np.int64), len(bits) - 1)
        km = np.concatenate([[0], np.cumsum(bits)])[k]
        f = np.where(bits[k] == 1, fm, fs)
        cycles = (fm * km + fs * (k - km)) / baud + f * (tt - k * ts) / rate
        sig[i0:i1] += amp * np.cos(2.0 * np.pi * (cycles - np.floor(cycles)))
    if sigma:
        sig += np.random.Generator(np.random.Philox(key=0x1E7E1 + seed)).standard_normal(n) * sigma
    sig += dc
    if dc_step is not None:
        sig[dc_step[0]:] += dc_step[1]
    out = np.clip(np.rint(sig), -32768, 32767).astype(np.int16)
    for at, piece in splice:
        out[at:at + len(piece)] = piece[: max(0, n - at)]
    return out


def event_bursts(t0, amp, baud=BAUD, rate=RATE, n_hdr=3, n_eom=3):
    """one SAME event from t0 (samples): header bursts then EOM bursts, 1 s gaps, at amplitude `amp`"""
    out, t = [], float(t0)
    for p in [HEADER] * n_hdr + [EOM] * n_eom:
        out.append((t, p, amp, baud))
        t += len(p) * 8 * rate / baud + rate
    return out


def worst_dc_pattern(sign=1):
    """the input that maximises |D| of the integer DC blocker: x[-15] at one rail, the 30 samples around it at the other"""
    hi, lo = (32767, -32768) if sign > 0 else (-32768, 32767)
    return np.array([lo] * 15 + [hi] + [lo] * 15, np.int16)


# ---------------------------------------------------------------------------------------------------------------------
# Helpers
# ---------------------------------------------------------------------------------------------------------------------
def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def builder(rate=RATE, samedec=True):
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


def state_words(blob):
    """[n_records, n_words] uint32 state words of an export (record layout: include/same_engine.h)"""
    head = np.frombuffer(blob[:HEADER_BYTES], "<u4")
    n, n_words, rec = int(head[4]), int(head[5]), int(head[8])
    recs = np.frombuffer(blob[HEADER_BYTES:HEADER_BYTES + n * rec], np.uint8).reshape(n, rec)
    return recs[:, RECORD_WORDS_AT:RECORD_WORDS_AT + 4 * n_words].copy().view("<u4")


def f32_bits(v):
    return np.float32(v).view(np.uint32)


def dc_words_reference(x, dc_len=16):
    """The 34 DC-blocker state words after the samples x (from a zero state), from the exact integer recursion of
    dcblock.rs:45-49,104-108: [ff window (last 16 samples, oldest first), fb window (last 16 moving sums S1 / 16),
    ff moving sum S1, fb moving sum S2 / 16] as f32 bits.  Every value is an integer / 16 below 2^24: exact in f32."""
    xp = np.concatenate([np.zeros(2 * dc_len, np.int64), np.asarray(x, np.int64)])
    c = np.concatenate([[0], np.cumsum(xp)])
    s1 = c[dc_len:] - c[:-dc_len]                       # s1[j] = sum xp[j .. j + 15]
    ff = xp[-dc_len:]
    fb = s1[-dc_len:]
    s2 = int(fb.sum())
    words = np.concatenate([f32_bits(ff.astype(np.float32)), f32_bits(fb.astype(np.float32) / np.float32(16)),
                            [f32_bits(np.float32(s1[-1])), f32_bits(np.float32(s2) / np.float32(16))]])
    return words.astype(np.uint32)


def dc_words_of(words, dc_len=16):
    """the same 34 words out of exported state words (same_params.h: dc_ff and dc_fb follow the scalars)"""
    ff0 = F_NUM_SCALARS
    return np.concatenate([words[..., ff0:ff0 + 2 * dc_len], words[..., [F_DC_FFSUM, F_DC_FBSUM]]], axis=-1)


def residue_chunks(n, seed, kmax):
    """chunk lengths 32 k + r summing to n, r cycling through 1..31 (every partial-chunk length of the fast kernels'
    DC blocker), k uniform in [0, kmax]"""
    rng = np.random.default_rng(seed)
    out, tot, r = [], 0, 1
    while tot < n:
        m = min(n - tot, 32 * int(rng.integers(0, kmax + 1)) + r)
        out.append(m)
        tot += m
        r = r % 31 + 1
    return out


def run_chunks(b, xs, lens, kernel=None, long_stream=None, trace=True, f32=False):
    """one engine over the streams xs in rounds of the given chunk lengths (each stream's chunk clipped to its own
    length): (events per stream, exported state after every round, engine)"""
    rx = b.build_batch(len(xs))
    if kernel is not None:
        rx.set_option("kernel", kernel)
    if long_stream is not None:
        rx.set_option("long_stream", long_stream)
    if trace:
        rx.enable_soft_trace(1 << 18)
    got, exports, pos = [[] for _ in xs], [], 0
    for m in lens:
        chunks = [x[pos:pos + m] for x in xs]
        for s, e in enumerate(rx.process_f32(chunks) if f32 else rx.process(chunks)):
            got[s].extend(e)
        exports.append(rx.export_streams())
        pos += m
    assert pos >= max(len(x) for x in xs)
    return got, exports, rx


def check_against_oracle(b, xs, got, rx, what, f32=False, trace=True):
    for s, x in enumerate(xs):
        o = oracle(b, x, f32)
        assert keys(got[s]) == keys(o.events()), f"{what}, stream {s}: events differ from the oracle"
        if trace:
            assert rx.read_soft_trace(s).tobytes() == o.soft_trace().tobytes(), f"{what}, stream {s}: soft-symbol trace differs"


# ---------------------------------------------------------------------------------------------------------------------
# a + b. Level x noise x offset sweep, every kernel, whole and in ragged chunks; DC state against the exact reference
# ---------------------------------------------------------------------------------------------------------------------
AMPS = [120.0, 250.0, 600.0, 2000.0, 8000.0, 16384.0, 32767.0, 65534.0]   # 65534: 32767 overdriven x2, then clipped
# (sigma, dc, dc step inside the second header burst, full-scale / worst-case DC / -32768 runs spliced in)
MIXES = [(0.0, 0.0, None, False), (2.0, 12000.0, None, False), (300.0, -20000.0, None, False), (3663.0, 0.0, None, False),
         (2.0, 0.0, 20000.0, False), (300.0, 0.0, None, True)]


def sweep_streams():
    xs, meta = [], []
    for ai, amp in enumerate(AMPS):
        for mi, (sigma, dc, step, extremes) in enumerate(MIXES):
            i = ai * len(MIXES) + mi
            n = (20 + (i * 7) % 21) * RATE
            bursts = event_bursts((1.0 + 0.37 * (i % 5)) * RATE, amp)
            splice = []
            if extremes:
                alt = np.tile(np.array([32767, -32768], np.int16), RATE // 2)      # full-scale: pins the gain at gmin
                splice = [(0, alt), (16 * RATE, worst_dc_pattern(1)), (16 * RATE + 400, worst_dc_pattern(-1)),
                          (17 * RATE, np.full(3000, -32768, np.int16)), (18 * RATE + 5, np.full(40, -32768, np.int16))]
            dstep = None if step is None else (int(bursts[1][0] + 0.5 * RATE), step)
            xs.append(render(n, bursts, sigma, seed=i, dc=dc, dc_step=dstep, splice=splice))
            meta.append((amp, sigma, dc, step, extremes))
    return xs, meta


def test_level_noise_offset_sweep_every_kernel_and_dc_state():
    _torch()
    b = builder()
    xs, meta = sweep_streams()
    assert len(xs) == 48
    n = max(len(x) for x in xs)
    gmin, gmax = f32_bits(b.config().agc_gain_min), f32_bits(b.config().agc_gain_max)
    seen_gmin = seen_gmax = False
    for chunking, lens in (("whole", [n]), ("ragged", residue_chunks(n, 11, 700))):
        assert chunking == "whole" or set(m % 32 for m in lens[:-1]) >= set(range(1, 32))
        ref_got, ref_exp, ref = run_chunks(b, xs, lens, kernel=1)
        check_against_oracle(b, xs, ref_got, ref, f"generic kernel, {chunking}")
        traces = [oracle(b, x).soft_trace().tobytes() for x in xs]
        pos = 0
        for k, m in enumerate(lens):                          # DC state of every stream after every chunk
            pos += m
            w = state_words(ref_exp[k])
            want = np.stack([dc_words_reference(x[:pos]) for x in xs])
            assert np.array_equal(dc_words_of(w), want), f"generic kernel, {chunking}: DC state after chunk {k}"
            seen_gmin |= bool(np.any(w[:, F_AGC_GAIN] == gmin))
            seen_gmax |= bool(np.any(w[:, F_AGC_GAIN] == gmax))
        for kernel in (2, 3, 4, 5, 6, 0):
            got, exp, rx = run_chunks(b, xs, lens, kernel=kernel)
            for k in range(len(lens)):
                assert exp[k] == ref_exp[k], f"kernel {kernel}, {chunking}: resident state differs after chunk {k}"
            for s in range(len(xs)):
                assert keys(got[s]) == keys(ref_got[s]), f"kernel {kernel}, {chunking}, stream {s}: events"
                assert rx.read_soft_trace(s).tobytes() == traces[s], f"kernel {kernel}, {chunking}, stream {s}: trace"
            if kernel == 3:
                assert rx.get_option("rollbacks") > 0
    assert seen_gmin and seen_gmax, (seen_gmin, seen_gmax)
    # the sweep decodes at the lowest amplitude and on clipped and overdriven bursts
    msgs = {}
    for x, (amp, sigma, dc, step, ext) in zip(xs, meta):
        if step is None and not ext:
            msgs.setdefault(amp, []).append(sum(1 for e in oracle(b, x).events() if e.kind == EV_SOM))
    assert min(msgs[AMPS[0]]) == 0 < max(msgs[AMPS[0]])
    assert max(msgs[32767.0]) > 0 and max(msgs[65534.0]) > 0


# ---------------------------------------------------------------------------------------------------------------------
# c. Long-stream path at quiet levels: verification stops, unverified spans
# ---------------------------------------------------------------------------------------------------------------------
def quiet_streams():
    out = {}
    for sigma in (300.0, 500.0, 1000.0, 1500.0, 3663.0):
        out[f"noise {sigma:g}"] = render(int((180 + sigma / 100) * RATE), sigma=sigma, seed=int(sigma))
    bursts = []
    for t0 in (20.0, 110.0, 200.0):
        bursts += event_bursts(t0 * RATE, 2000.0)
    out["bursts 2000 over 500"] = render(240 * RATE + 333, bursts, 500.0, seed=7)
    return out


def test_long_stream_path_at_quiet_levels():
    _torch()
    b = builder()
    rng = np.random.default_rng(23)
    for name, x in quiet_streams().items():
        ragged = []
        while sum(ragged) < len(x):
            ragged.append(int(rng.integers(65536, 3 * 65536)))
        for chunking, lens in (("whole", [len(x)]), ("ragged", ragged)):
            got, exp, rx = run_chunks(b, [x], lens, long_stream=1)
            ref_got, ref_exp, _ = run_chunks(b, [x], lens, long_stream=0)
            check_against_oracle(b, [x], got, rx, f"long path, {name}, {chunking}")
            for k in range(len(lens)):
                assert exp[k] == ref_exp[k], f"{name}, {chunking}: state differs from long_stream = 0 after chunk {k}"
            passes, spans = rx.get_option("long_stream_passes"), rx.get_option("long_stream_fallback_spans")
            starts = np.cumsum([0] + lens[:-1])
            big = [m for m, s0 in zip(lens, starts) if min(m, len(x) - s0) >= 65536]   # submits the long path takes
            if name == "noise 500":           # hand-overs fail: the path stops at a verified end again and again
                assert passes >= 2 * len(big) and spans >= 1, (chunking, passes, spans)
            if name == "noise 3663":          # every hand-over verifies: one pass per chunk, no fallback
                assert passes == len(big) and spans == 0, (chunking, passes, spans)
            if name.startswith("bursts"):
                assert any(e.kind == EV_SOM for e in got[0]) and spans >= 1


# ---------------------------------------------------------------------------------------------------------------------
# d. f32 ingest at scale extremes (rate-generic kernel)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [22050, 44100])
@pytest.mark.parametrize("samedec", [True, False])
def test_f32_ingest_at_scale_extremes(rate, samedec):
    _torch()
    b = builder(rate, samedec)
    if rate == RATE:
        base = [load_golden_recording(n) for n in NAMES]
    else:
        base = [render(14 * rate, event_bursts(1.0 * rate, 16384.0, rate=rate), 2000.0, seed=3, rate=rate)]
    seen_sub = False
    for scale in (1e-42, 1e-20, 1e30):
        xs = [(x.astype(np.float32) * np.float32(scale)).astype(np.float32) for x in base]
        assert all(np.all(np.isfinite(x)) for x in xs)
        seen_sub |= any(np.any((x != 0) & (np.abs(x) < np.finfo(np.float32).tiny)) for x in xs)
        n = max(len(x) for x in xs)
        for chunking, lens in (("whole", [n]), ("chunked", residue_chunks(n, 5, 3000))):
            got, _, rx = run_chunks(b, xs, lens, f32=True)
            check_against_oracle(b, xs, got, rx, f"f32 x {scale:g} at {rate} Hz, {chunking}", f32=True)
    assert seen_sub


# ---------------------------------------------------------------------------------------------------------------------
# e. Off-rate symbols: the timing loop at its period clamp
# ---------------------------------------------------------------------------------------------------------------------
DEVS = [-0.02, -0.01, -0.005, 0.005, 0.01, 0.02]


def off_rate_streams(rate):
    return [render(16 * rate, event_bursts(1.0 * rate, 12000.0, baud=BAUD * (1 + d), rate=rate, n_eom=1), 300.0,
                   seed=100 + i, rate=rate) for i, d in enumerate(DEVS)]


@pytest.mark.parametrize("rate,kernels", [(22050, (1, 2, 3, 4, 5, 6, 0)), (48000, (1,))])
def test_off_rate_symbols_drive_the_period_to_its_clamp(rate, kernels):
    _torch()
    b = builder(rate)
    xs = off_rate_streams(rate)
    lens = residue_chunks(16 * rate, 9, 60)
    d = b.build_batch(1).derived()
    pmin, pmax = f32_bits(d["period_min"]), f32_bits(d["period_max"])
    ref_exp = None
    for kernel in kernels:
        got, exp, rx = run_chunks(b, xs, lens, kernel=kernel)
        if ref_exp is None:
            check_against_oracle(b, xs, got, rx, f"off-rate symbols at {rate} Hz")
            ref_exp, ref_got = exp, got
            pavg = np.stack([state_words(e)[:, F_PAVG] for e in exp])     # [chunk, stream]
            for s, dev in enumerate(DEVS):
                if abs(dev) == 0.02:
                    assert np.any(pavg[:, s] == (pmin if dev > 0 else pmax)), f"deviation {dev}: pavg never at its clamp"
            continue
        for k in range(len(lens)):
            assert exp[k] == ref_exp[k], f"kernel {kernel}, {rate} Hz: resident state differs after chunk {k}"
        assert [keys(g) for g in got] == [keys(g) for g in ref_got], f"kernel {kernel}: events"

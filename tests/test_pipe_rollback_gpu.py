"""GPU tests of the pipelined kernel's roll-back (kernel 3, same_rx_pipe_kernel): its timing warp runs ahead of the
symbol stages and resumes a stream from a symbol whose symbol stages changed the timing loop's state (sync found: AGC
and bandwidth locked; end of a burst or a dropped carrier: timing loop reset).  After every chunk the resident state
of every stream (export_streams) must equal the rate-generic kernel's on the same chunks, and the events and the
soft-symbol trace must equal the CPU oracle's.  Each case also checks that roll-backs happened, so that it exercises
the roll-back path rather than only the speculation."""
import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle, load_golden_recording
from oracle.pyoracle import OracleConfig
from sameold_b200 import synth

pytestmark = pytest.mark.gpu

RATE = 22050
NAMES = ["long_message", "npt", "two_and_two"]
EV_READING, EV_BURST, EV_SOM = 2, 3, 18
SYM = RATE / 520.83


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def builder():
    return sb.SameReceiverBuilder.samedec(RATE)


def ocfg(b) -> OracleConfig:
    c, o = b.config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    return o


def oracle(b, rec, trace=False):
    o = Oracle(ocfg(b))
    if trace:
        o.enable_trace()
    o.process_s16(rec)
    return o


def keys(evs):
    return [e.key() for e in evs]


def rounds_from_cuts(recs, cuts):
    """per-round chunk lengths from per-stream sorted cut positions (each stream ends at its own length)"""
    per = []
    for r, c in zip(recs, cuts):
        pts = sorted({int(x) for x in c if 0 < x < len(r)} | {len(r)})
        per.append(np.diff([0] + pts))
    n = max(len(x) for x in per)
    return [[int(x[k]) if k < len(x) else 0 for x in per] for k in range(n)]


def lockstep(b, recs, rounds, trace=False, check_every=1):
    """The pipelined and the generic kernel over the same chunks: resident state compared after every `check_every`-th
    chunk and at the end, events and trace against the oracle.  Returns the pipelined engine's roll-back count."""
    ns = len(recs)
    pipe, ref = b.build_batch(ns), b.build_batch(ns)
    pipe.set_option("kernel", 3)
    ref.set_option("kernel", 1)
    if trace:
        for rx in (pipe, ref):
            rx.enable_soft_trace(1 << 18)
    pos = [0] * ns
    got = [[] for _ in range(ns)]
    for k, lens in enumerate(rounds):
        chunks = [recs[s][pos[s]:pos[s] + lens[s]] for s in range(ns)]
        pos = [p + n for p, n in zip(pos, lens)]
        for s, e in enumerate(pipe.process(chunks)):
            got[s].extend(e)
        ref.process(chunks)
        if k % check_every == 0 or k == len(rounds) - 1:
            assert pipe.export_streams() == ref.export_streams(), f"resident state differs after chunk {k}"
    assert pos == [len(r) for r in recs]
    for s in range(ns):
        o = oracle(b, recs[s], trace)
        assert keys(got[s]) == keys(o.events()), f"stream {s}: events differ from the oracle"
        if trace:
            t, ot = pipe.read_soft_trace(s), o.soft_trace()
            assert t.tobytes() == ot.tobytes(), f"stream {s}: soft-symbol trace differs from the oracle"
    return pipe.get_option("rollbacks")


def event_samples(b, rec, kinds):
    return [e.sample for e in oracle(b, rec).events() if e.kind in kinds]


def test_tiny_chunks_with_trace():
    """Chunks of 1-64 samples cut T's lead all the time; the soft-symbol trace is on."""
    _torch()
    b = builder()
    recs = [load_golden_recording(n) for n in NAMES]
    rng = np.random.default_rng(5)
    cut = np.cumsum(rng.integers(1, 65, max(len(r) for r in recs) // 16))
    rounds = rounds_from_cuts(recs, [cut] * len(recs))
    assert lockstep(b, recs, rounds, trace=True, check_every=97) > 0


def test_chunk_boundaries_near_sync_and_burst_ends():
    """Chunk boundaries within T's lead (a few symbols) before and after every link event: the symbol that starts or
    ends a burst is confirmed in one launch and rolled back to in the next."""
    _torch()
    b = builder()
    recs = [load_golden_recording(n) for n in NAMES]
    recs += [synth.render_numpy(synth.plan_stream(40 + i, seconds=40.0), 40 * RATE) for i in range(3)]
    cuts = []
    for r in recs:
        c = []
        for x in event_samples(b, r, (1, EV_READING, EV_BURST, 0)):
            c += [x + d for d in (-311, -42, -1, 0, 1, 21, 43, 170)]
        cuts.append(c)
    assert lockstep(b, recs, rounds_from_cuts(recs, cuts), trace=True) > 0


def _plan(starts, payloads, seed, foff=1.5):
    return synth.StreamPlan("", list(starts), list(payloads), foff, seed)


def test_back_to_back_bursts_and_dropped_carrier():
    """Bursts with almost no gap between them, and a carrier that stops in the middle of a burst (silence and noise)."""
    _torch()
    b = builder()
    hdr = synth.PREAMBLE + b"ZCZC-WXR-TOR-029165-029169+0030-1051700-KEAX/NWS-"
    eom = synth.PREAMBLE + b"NNNN"
    recs = []
    for gap in (0.0, 3.0, 40.0):   # in samples
        t, starts, pays = 0.5 * RATE, [], []
        for p in (hdr, hdr, hdr, eom, eom, eom):
            starts.append(t); pays.append(p); t += len(p) * 8 * SYM + gap
        recs.append(synth.render_numpy(_plan(starts, pays, 77 + int(gap)), int(t + RATE)))
    base = synth.render_numpy(synth.plan_stream(9, seconds=40.0), 40 * RATE)
    p9 = synth.plan_stream(9, seconds=40.0)
    for k, fill in enumerate(("zero", "noise")):
        r = base.copy()
        s0 = int(p9.burst_starts[1 + k] + 0.4 * len(p9.burst_payloads[1 + k]) * 8 * SYM)
        r[s0:s0 + RATE // 2] = 0 if fill == "zero" else np.random.default_rng(k).normal(0, 300, RATE // 2).astype(np.int16)
        recs.append(r)
    rng = np.random.default_rng(3)
    cuts = [np.cumsum(rng.integers(1, 9000, 200)) for _ in recs]
    assert lockstep(b, recs, rounds_from_cuts(recs, cuts), check_every=3) > 0


def test_forced_end_of_message():
    """A header without EOM bursts: the forced EOM 135 s later, with the timing warp running ahead over the silence."""
    _torch()
    b = builder()
    p = synth.plan_stream(21, seconds=180.0)
    recs = [synth.render_numpy(_plan(p.burst_starts[:3], p.burst_payloads[:3], p.seed), 180 * RATE)]
    p2 = synth.plan_stream(22, seconds=180.0)
    recs.append(synth.render_numpy(_plan(p2.burst_starts[:2], p2.burst_payloads[:2], p2.seed), 175 * RATE + 777))
    rng = np.random.default_rng(8)
    cuts = [np.cumsum(rng.integers(1, 3 * RATE, 200)) for _ in recs]
    assert lockstep(b, recs, rounds_from_cuts(recs, cuts), check_every=5) > 0
    assert any(e.kind == 19 for e in oracle(b, recs[0]).events())   # the forced EOM is there to be compared


def test_low_snr_corpus_ragged_lengths():
    """1024 streams at 0-3 dB SNR (false acquires: roll-backs on many lanes of one warp at different times), ragged
    lengths within every block, chunked: every stream's state and events equal to the generic kernel's; a sample of
    streams against the oracle."""
    torch = _torch()
    b = builder()
    ns, secs = 1024, 20.0
    n = int(secs * RATE)
    stride = (n + 7) // 8 * 8
    buf = torch.empty((ns, stride), dtype=torch.int16, device="cuda")
    plans = synth.plan_corpus(ns, RATE, secs, first_stream=3000)
    for q in range(4):   # 0, 1, 2, 3 dB: one quarter of the streams each
        sig = synth.NOISE_SIGMA * np.sqrt(10.0) / np.sqrt(10.0 ** (q / 10.0))
        part = buf[q * ns // 4:(q + 1) * ns // 4]
        synth.generate_on_device(plans[q * ns // 4:(q + 1) * ns // 4], part.data_ptr(), stride, n, RATE, noise_sigma=sig)
    host = buf.cpu().numpy()
    lengths = (n - (np.arange(ns) * 7919) % 60000).astype(np.uint32)
    offsets = np.arange(ns, dtype=np.uint64) * np.uint64(stride)
    pipe, ref = b.build_batch(ns), b.build_batch(ns)
    pipe.set_option("kernel", 3)
    ref.set_option("kernel", 1)
    got = [[] for _ in range(2)]
    lo = 0
    for step in (5 * RATE + 13, 31, 7 * RATE + 1, n):
        hi = min(lo + step, n)
        ln = np.clip(lengths.astype(np.int64) - lo, 0, hi - lo).astype(np.uint32)
        for i, rx in enumerate((pipe, ref)):
            rx.submit_device(buf.data_ptr() + 2 * lo, ns * stride - lo, offsets, ln)
            rx.sync()
            got[i].append(rx.drain_by_stream())
        assert pipe.export_streams() == ref.export_streams(), f"resident state differs after the chunk at {lo}"
        lo = hi
        if lo >= n:
            break
    ev = [[sum((g[k][s] for k in range(len(g))), []) for s in range(ns)] for g in got]
    for s in range(ns):
        assert keys(ev[0][s]) == keys(ev[1][s]), f"stream {s}: pipelined and generic kernels differ"
    for s in (0, 1, 31, 255, 256, 600, 1023):
        o = Oracle(ocfg(b))
        o.process_s16(host[s, :lengths[s]])
        assert keys(ev[0][s]) == keys(o.events()), f"stream {s} against the oracle"
    rb = pipe.get_option("rollbacks")
    assert rb >= ns // 4, rb


def test_import_mid_burst_and_mid_pending_hold():
    """A stream exported in the middle of a burst or while a header is held, imported into a slot of a 64-stream
    pipelined engine, continues exactly as the oracle's run over the whole recording."""
    _torch()
    b = builder()
    recs = [load_golden_recording(n) for n in NAMES]
    checked = 0
    for r in recs:
        evs = oracle(b, r).events()
        reading = [e.sample for e in evs if e.kind == EV_READING]
        bursts = [e.sample for e in evs if e.kind == EV_BURST]
        for split in (reading[0] + 3000, bursts[0] + 4000):
            src = b.build_batch(1)
            src.set_option("kernel", 3)
            first = src.process([r[:split]])[0]
            dst = b.build_batch(64)
            dst.set_option("kernel", 3)
            dst.import_streams(src.export_streams(), [37])
            rest = dst.process([r[split:] if i == 37 else r[:0] for i in range(64)])[37]
            assert keys(first + rest) == keys(evs), f"split at {split}"
            assert dst.get_option("rollbacks") > 0
            checked += 1
    assert checked == 2 * len(recs)

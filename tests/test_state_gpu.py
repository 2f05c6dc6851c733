"""GPU tests of the portable stream state (same_engine_export_streams / same_engine_import_streams and the layers above
them): a stream exported from one engine and imported into another continues bit-exactly where it stopped — every
event equal to the CPU oracle's run over the whole recording (kind, sample counter, symbol count, bytes, parity and
voting counts) and the per-stream sequence numbers continuous.  Split points come from the oracle's own event list, so
each one falls into the receiver phase it names."""
import os
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle, decode_batch_events, load_golden_recording
from oracle.pyoracle import OracleConfig
from sameold_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["long_message", "npt", "two_and_two"]
HDR = 2224
F_SQ_HEAD = 33
EV_SEARCHING, EV_READING, EV_BURST, EV_SOM, EV_EOM = 1, 2, 3, 18, 19


def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def ocfg(builder) -> OracleConfig:
    c, o = builder.config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    return o


def keys(evs):
    return [e.key() for e in evs]


def oracle_run(builder, parts, flush=True, trace=False):
    """events of the oracle over the concatenation of `parts` (s16 arrays, or ('f32', array))"""
    o = Oracle(ocfg(builder))
    if trace:
        o.enable_trace()
    for p in parts:
        if isinstance(p, tuple):
            o.process_f32(p[1])
        else:
            o.process_s16(p)
    if flush:
        o.flush_samedec()
    return o


def recordings():
    out = {n: load_golden_recording(n) for n in NAMES}
    for i in (3, 11):
        out[f"synth{i}"] = synth.render_numpy(synth.plan_stream(i, seconds=60.0), 60 * 22050)
    return out


_RECS = None


def recs():
    global _RECS
    if _RECS is None:
        _RECS = recordings()
    return _RECS


def split_points(builder, rec):
    """{phase: sample index} from the oracle's events over the whole recording"""
    evs = oracle_run(builder, [rec]).events()
    pts = {}
    if evs:
        pts["before_sync"] = max(1, evs[0].sample - 2000)
    for a, b in zip(evs, evs[1:]):
        if a.kind == EV_READING and b.kind == EV_BURST:
            pts.setdefault("mid_burst", (a.sample + b.sample) // 2)
    for i, e in enumerate(evs):
        if e.kind == EV_SOM:
            last_burst = max((x.sample for x in evs[:i] if x.kind == EV_BURST), default=0)
            pts.setdefault("pending_hold", (last_burst + e.sample) // 2)
            nxt = next((x.sample for x in evs[i + 1:] if x.kind == EV_EOM), e.sample + 135 * 22050)
            pts.setdefault("eom_window", min(e.sample + 3 * 22050, (e.sample + nxt) // 2))
    return {k: v for k, v in pts.items() if 0 < v < rec.size}


def test_continuation_across_engines_at_every_phase():
    """A runs to the split and exports, then is destroyed; a fresh B imports, runs the rest and the EOF flush."""
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    phases_seen = set()
    for name, rec in recs().items():
        want = keys(oracle_run(b, [rec]).events())
        for phase, cut in split_points(b, rec).items():
            a = b.build_batch(1)
            a.submit([rec[:cut]])
            a.sync()
            ev_a, pay_a = a.drain_raw()
            data = a.export_streams()
            n_a = a.input_sample_counters().copy()
            a.close()
            rx = sb.SameBatchReceiver.from_state(data)
            assert np.array_equal(rx.input_sample_counters(), n_a)
            rx.submit([rec[cut:]])
            rx.sync()
            ev_b, pay_b = rx.drain_raw()
            tail = rx.flush_samedec()[0]
            got = sb.SameBatchReceiver.events_from_raw(ev_a, pay_a) + sb.SameBatchReceiver.events_from_raw(ev_b, pay_b) + tail
            assert keys(got) == want, f"{name} split {phase} at {cut}"
            seq = np.concatenate([ev_a["seq"], ev_b["seq"]])
            assert np.array_equal(seq, np.arange(seq.size)), f"{name} {phase}: seq not continuous"
            phases_seen.add(phase)
    assert phases_seen == {"before_sync", "mid_burst", "pending_hold", "eom_window"}


def test_other_geometry_pipelined_kernel_and_long_stream_path():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    names = ["long_message", "npt", "two_and_two"]
    rs = [recs()[n] for n in names]
    cuts = [split_points(b, r)["mid_burst"] for r in rs]
    src = b.build_batch(3)
    pre = src.process([r[:c] for r, c in zip(rs, cuts)])
    data = src.export_streams()
    # into ids [4095, 17, 2048] of a 4096-stream engine (pipelined kernel)
    big = b.build_batch(4096)
    assert big.get_option("kernel_selected") == 3
    ids = [4095, 17, 2048]
    big.import_streams(data, ids)
    chunks = [None] * 4096
    for i, s in enumerate(ids):
        chunks[s] = rs[i][cuts[i]:]
    evs = big.process(chunks)
    for i, s in enumerate(ids):
        o = oracle_run(b, [rs[i]], flush=False)
        assert keys(pre[i] + evs[s]) == keys(o.events()), names[i]
    # one stream, chunks >= 65536 samples: the long-stream path
    for i in range(3):
        one = b.build_batch(1)
        one.import_streams(src.export_streams([i]))
        rest = rs[i][cuts[i]:]
        if rest.size < 65536:
            rest = np.concatenate([rest, np.zeros(65536 - rest.size, np.int16)])
        ev = one.process([rest])[0]
        assert one.get_option("long_stream_passes") > 0
        o = oracle_run(b, [rs[i], np.zeros(max(0, 65536 - (rs[i].size - cuts[i])), np.int16)], flush=False)
        assert keys(pre[i] + ev) == keys(o.events()), names[i]


def test_export_changes_nothing_and_round_trips():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    rs = [recs()["two_and_two"], recs()["synth3"]]
    cut = [split_points(b, r)["pending_hold"] for r in rs]
    x, y = b.build_batch(2), b.build_batch(2)
    x.submit([r[:c] for r, c in zip(rs, cut)])
    y.submit([r[:c] for r, c in zip(rs, cut)])
    x.sync()
    y.sync()
    data = x.export_streams()                    # pending events stay pending
    for rx in (x, y):
        rx.submit([r[c:] for r, c in zip(rs, cut)])
        rx.sync()
    ex, px = x.drain_raw()
    ey, py = y.drain_raw()
    assert np.array_equal(ex, ey) and np.array_equal(px, py)
    assert x.export_streams() == y.export_streams()
    # export -> import -> export with the same ids: byte-identical; counters follow
    z = b.build_batch(2)
    z.import_streams(data)
    assert z.export_streams() == data
    w = b.build_batch(5)
    w.import_streams(data, [3, 1])
    assert _bodies(w.export_streams([3, 1])) == _bodies(data)
    c = w.input_sample_counters()
    assert [int(c[3]), int(c[1])] == [int(cut[0]), int(cut[1])]


def _records(data):
    n = struct.unpack_from("<I", data, 16)[0]
    rb = struct.unpack_from("<I", data, 32)[0]
    return [bytearray(data[HDR + i * rb: HDR + (i + 1) * rb]) for i in range(n)]


def _bodies(data):
    return [bytes(r[4:-4]) for r in _records(data)]


def test_receiver_clone():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    rec = recs()["npt"]
    other = recs()["synth11"]
    cut = split_points(b, rec)["pending_hold"]
    r = b.build()
    pre = list(r.iter_events(rec[:cut]))
    c = r.clone()
    assert c.input_sample_counter() == r.input_sample_counter() == cut
    want = keys(oracle_run(b, [rec], flush=False).events())
    assert keys(pre + list(r.iter_events(rec[cut:]))) == want
    assert keys(pre + list(c.iter_events(rec[cut:]))) == want
    # different remainders: no shared state
    r2 = b.build()
    list(r2.iter_events(rec[:cut]))
    c2 = r2.clone()
    ev_r = list(r2.iter_events(rec[cut:]))
    ev_c = list(c2.iter_events(other))
    assert keys(pre + ev_r) == want
    assert keys(pre + ev_c) == keys(oracle_run(b, [rec[:cut], other], flush=False).events())


def test_f32_state_travels_with_the_records():
    _torch()
    lib_default = sb.SameReceiverBuilder(22050)
    rec = recs()["npt"]
    f = rec.astype(np.float32) / 32768.0
    cut = split_points(lib_default, rec)["mid_burst"]
    a = lib_default.build_batch(1)
    pre = a.process_f32([f[:cut]])[0]
    data = a.export_streams()
    assert _records(data)[0][4] & 1
    rx = sb.SameBatchReceiver.from_state(data)
    assert rx.get_option("kernel_selected") == 1
    post = rx.process_f32([f[cut:]])[0]
    o = oracle_run(lib_default, [("f32", f)], flush=False)
    assert keys(pre + post) == keys(o.events())
    # s16-only records keep the fast kernel
    s = sb.SameReceiverBuilder.samedec(22050)
    q = s.build_batch(1)
    q.process([rec[:cut]])
    fresh = s.build_batch(1)
    k0 = fresh.get_option("kernel_selected")
    assert k0 != 1
    fresh.import_streams(q.export_streams())
    assert fresh.get_option("kernel_selected") == k0


def test_snapshot_restore_keeps_the_f32_flag():
    """f32 submit, snapshot, reset(all), restore, s16 submit: the s16 part must still run the literal f32 DC blocker
    on the non-integer state the f32 part left."""
    _torch()
    b = sb.SameReceiverBuilder(22050)
    rec = recs()["npt"]
    cut = split_points(b, rec)["before_sync"]
    f = rec[:cut].astype(np.float32) / 32768.0 + np.float32(0.3)
    rx = b.build_batch(1)
    pre = rx.process_f32([f])[0]
    snap = rx.snapshot()
    try:
        rx.reset()
        rx.restore(snap)
    finally:
        rx.free_snapshot(snap)
    assert rx.get_option("kernel_selected") == 1
    post = rx.process([rec[cut:]])[0]
    o = oracle_run(b, [("f32", f), rec[cut:]], flush=False)
    assert keys(pre + post) == keys(o.events())


def _target_engine(b):
    rx = b.build_batch(4)
    rx.process([recs()[n][:200000] for n in NAMES] + [recs()["synth3"][:200000]])
    return rx


def _reference_continuation(rx, b):
    return rx.process([recs()[n][200000:400000] for n in NAMES] + [recs()["synth3"][200000:400000]])


def _rejections():
    samedec = sb.SameReceiverBuilder.samedec(22050)

    def export_from(builder, rate_rec=None):
        a = builder.build_batch(1)
        a.process([recs()["npt"][:100000]])
        return a.export_streams()

    good = export_from(samedec)
    one = bytes(good)

    def crc_fixed(buf, i, off, val):
        recs_ = _records(buf)
        r = recs_[i]
        struct.pack_into("<I", r, off, val)
        struct.pack_into("<I", r, len(r) - 4, zlib.crc32(bytes(r[:-4])))
        out = bytearray(buf)
        rb = len(r)
        out[HDR + i * rb: HDR + (i + 1) * rb] = r
        return bytes(out)

    flipped = bytearray(one)
    flipped[HDR + 1000] ^= 0x10
    bad_magic = bytearray(one)
    bad_magic[0] ^= 1
    two = samedec.build_batch(2)
    two.process([recs()["npt"][:100000], recs()["two_and_two"][:100000]])
    two_recs = two.export_streams()
    return [
        ("rate", export_from(sb.SameReceiverBuilder.samedec(44100)), [0], 2),
        ("eq_off", export_from(sb.SameReceiverBuilder.samedec(22050).without_adaptive_equalizer()), [0], 2),
        ("agc_limits", export_from(sb.SameReceiverBuilder(22050)), [0], 2),
        ("truncated", one[:-1], [0], 1),
        ("bad_magic", bytes(bad_magic), [0], 1),
        ("n_mismatch", two_recs, [0], 1),
        ("duplicate_ids", two_recs, [1, 1], 1),
        ("id_out_of_range", one, [4], 1),
        ("crc", bytes(flipped), [2], 1),
        ("sq_head", crc_fixed(one, 0, 8 + 4 * F_SQ_HEAD, 64), [2], 1),
    ]


def test_rejected_import_leaves_every_stream_untouched():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    ref = _target_engine(b)
    want = keys(sum(_reference_continuation(ref, b), []))
    for what, data, ids, code in _rejections():
        rx = _target_engine(b)
        before = rx.export_streams()
        with pytest.raises(sb.SameEngineError) as ei:
            rx.import_streams(data, ids)
        assert ei.value.code == code, (what, str(ei.value))
        assert rx.export_streams() == before, what
        assert keys(sum(_reference_continuation(rx, b), [])) == want, what


def test_import_drops_target_events_only_and_restarts_the_trace():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    rec = recs()["npt"]
    cut = split_points(b, rec)["mid_burst"]
    src = b.build_batch(1)
    src.process([rec[:cut]])
    data = src.export_streams()
    rx = b.build_batch(3)
    rx.enable_soft_trace(1 << 17)
    rx.submit([rec, rec, rec])
    rx.sync()                                     # events of all three streams are pending
    rx.import_streams(data, [1])
    evs = rx.drain_by_stream()
    full = keys(oracle_run(b, [rec], flush=False).events())
    assert keys(evs[0]) == full and keys(evs[2]) == full and evs[1] == []
    rx.read_soft_trace(1)                         # rewinds; the import already emptied it
    rx.enable_soft_trace(1 << 17)
    rx.import_streams(data, [1])
    assert rx.read_soft_trace(1).size == 0
    post = rx.process([None, rec[cut:], None])[1]
    t = rx.read_soft_trace(1)
    o = oracle_run(b, [rec], flush=False, trace=True)
    ot = o.soft_trace()
    ot = ot[ot["sample"] > cut]
    assert len(t) == len(ot) and len(t) > 0
    assert np.array_equal(t["sample"], ot["sample"])
    assert np.array_equal(t["zero"].view(np.uint32), ot["zero"].view(np.uint32))
    assert np.array_equal(t["sym"].view(np.uint32), ot["sym"].view(np.uint32))
    assert keys(src.process([rec[cut:]])[0]) == keys(post)


def test_multi_receiver_export_and_permuted_import():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    rs = [recs()[n] for n in ("long_message", "npt", "two_and_two", "synth3")]
    cuts = [split_points(b, r)["mid_burst"] for r in rs]
    m2 = b.build_multi(4, [0, 0])                 # shards: streams 0-1 | 2-3
    pre = m2.process([r[:c] for r, c in zip(rs, cuts)])
    gids = [3, 0, 2]
    data = m2.export_streams(gids)
    m3 = b.build_multi(6, [0, 0, 0])              # shards: 0-1 | 2-3 | 4-5
    tgt = [5, 1, 3]
    m3.import_streams(data, tgt)
    assert _bodies(m3.export_streams(tgt)) == _bodies(data)
    chunks = [None] * 6
    for g, t in zip(gids, tgt):
        chunks[t] = rs[g][cuts[g]:]
    evs = m3.process(chunks)
    for g, t in zip(gids, tgt):
        assert keys(pre[g] + evs[t]) == keys(oracle_run(b, [rs[g]], flush=False).events()), g


def test_state_survives_a_process_restart(tmp_path):
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    rec = recs()["long_message"]
    cut = split_points(b, rec)["pending_hold"]
    out = tmp_path / "state.bin"
    ev_file = tmp_path / "events.npy"
    script = f"""
import numpy as np, sameold_b200 as sb
from oracle import load_golden_recording
rec = load_golden_recording("long_message")
r = sb.SameReceiverBuilder.samedec(22050).build()
evs = list(r.iter_events(rec[:{cut}]))
open({str(out)!r}, "wb").write(r.export_state())
np.save({str(ev_file)!r}, np.array([e.sample for e in evs], np.int64))
"""
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-c", script], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    rx = sb.SameBatchReceiver.from_state(out.read_bytes())
    post = rx.process([rec[cut:]])[0] + rx.flush_samedec()[0]
    want = oracle_run(b, [rec]).events()
    n_pre = np.load(ev_file).size
    assert [e.sample for e in want[:n_pre]] == list(np.load(ev_file))
    assert keys(post) == keys(want[n_pre:])


def test_across_devices():
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU: export on device 0, import on device 1 needs two")
    b = sb.SameReceiverBuilder.samedec(22050)
    rec = recs()["npt"]
    cut = split_points(b, rec)["pending_hold"]
    r = b.build(device=0)
    pre = list(r.iter_events(rec[:cut]))
    c = r.clone(device=1)
    assert keys(pre + list(c.iter_events(rec[cut:]))) == keys(oracle_run(b, [rec], flush=False).events())


def test_scale_16384_streams():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    n, distinct, sec = 16384, 61, 10
    rate = 22050
    base = np.stack([synth.render_numpy(synth.plan_stream(100 + i, seconds=2 * sec), 2 * sec * rate) for i in range(distinct)])
    rows = np.arange(n) % distinct

    def feed(rx, t0, t1):
        out = [[] for _ in range(n)]
        for c0 in range(t0, t1, rate):
            evs = rx.process(np.ascontiguousarray(base[rows, c0:min(c0 + rate, t1)]))
            for s in range(0, n, 16):
                out[s] += evs[s]
        return out

    a = b.build_batch(n)
    pre = feed(a, 0, sec * rate)
    data = a.export_streams()
    assert len(data) == HDR + n * 4032
    a.close()
    rx = b.build_batch(n)
    rx.import_streams(data)
    post = feed(rx, sec * rate, 2 * sec * rate)
    ev, pay, _ = decode_batch_events(ocfg(b), base, os.cpu_count() or 4)
    want = [[] for _ in range(distinct)]
    for e in sb.SameBatchReceiver.events_from_raw(ev, pay):
        want[e.stream].append(e)
    for s in range(0, n, 16):
        assert keys(pre[s] + post[s]) == keys(want[rows[s]]), s
    # a contiguous range and a random permutation
    ids = np.arange(5000, 9000, dtype=np.uint32)
    part = rx.export_streams(ids)
    c = b.build_batch(n)
    c.import_streams(part, ids)
    assert c.export_streams(ids) == part
    perm = np.random.default_rng(7).permutation(n).astype(np.uint32)
    d = b.build_batch(n)
    d.import_streams(data, perm)
    assert _bodies(d.export_streams(perm)) == _bodies(data)

"""Interleaved ingest on one GPU: the deinterleave kernel alone, the end-to-end host path, and the host cost it removes.

    python tools/ingest.py [--out results.jsonl]

One JSON line per measurement on stdout (and appended to --out if given), each with the card's name, power limit and max SM clock read in the same run.

  kernel   same_ingest_kernel<fmt> alone on device-resident frames of >= --gb GiB (beyond the 126 MB L2), for every
           format and n_channels in {1, 2, 8, 64, 4096}, every column mapped: GB/s of bytes read + bytes written, CUDA
           events over --reps launches, against a device-to-device cudaMemcpyAsync of the input size in the same run
           (2 x size bytes moved).
  e2e      the config-3 corpus (4096 streams x 60 s, 22 050 Hz) from pinned host memory, in --chunks time-chunks:
           interleaved s16 frames through same_engine_submit_interleaved against the same samples through
           same_engine_submit_s16_2d, the two arms alternating on one engine; events must be identical.  audio-s/s from
           the engine's device stopwatch, and each arm's H2D rate as a fraction of same_h2d_probe run with that arm's
           copy geometry (planar: strided rows; interleaved: one flat run per chunk).
  numpy    the host deinterleave this replaces, np.ascontiguousarray(frames.T), on --host-gb GiB blocks (n_channels
           from 2 on: one channel needs none).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import sameold_b200 as sb  # noqa: E402
from sameold_b200 import _lib, synth  # noqa: E402

FORMATS = {"s16": (0, 2, 2), "s24": (1, 3, 4), "s32": (2, 4, 4), "f32": (3, 4, 4)}   # code, bytes in, bytes out
CHANNELS = [1, 2, 8, 64, 4096]


def card():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:   # reported, not guessed
        out["power_limit"] = f"unread: {e}"
    return out


def kernel_leg(args, info, emit):
    import torch
    lib = _lib.load()
    launch = lib.same_launch_ingest   # the launcher same_engine_submit_interleaved uses (same_internal.h)
    launch.restype = C.c_int
    launch.argtypes = [C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    st = torch.cuda.current_stream()
    for name, (code, isz, osz) in FORMATS.items():
        for nc in CHANNELS:
            n_frames = min(1 << 30, int(args.gb * (1 << 30)) // (nc * isz))
            src = torch.randint(0, 256, (n_frames * nc * isz,), dtype=torch.uint8, device="cuda")
            dpitch = (n_frames + 7) // 8 * 8
            dst = torch.empty(nc * dpitch * osz, dtype=torch.uint8, device="cuda")
            rows = torch.arange(nc, dtype=torch.int32, device="cuda")
            cp = torch.empty_like(src)

            def run():
                rc = launch(code, src.data_ptr(), nc * isz, nc, n_frames, rows.data_ptr(), dst.data_ptr(), dpitch, st.cuda_stream)
                assert rc == 0, rc

            def timed(fn):
                fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.reps):
                    fn()
                b.record()
                b.synchronize()
                return a.elapsed_time(b) / args.reps

            ms = timed(run)
            ms_copy = timed(lambda: cp.copy_(src))
            moved = n_frames * nc * (isz + osz)
            gbs, copy_gbs = moved / ms / 1e6, 2 * src.numel() / ms_copy / 1e6
            # spot check: column nc-1 of the first frames, as the engine reads it
            if name == "s16":
                want = src[: 64 * nc * 2].view(torch.int16).view(64, nc)[:, nc - 1]
                got = dst.view(torch.int16)[(nc - 1) * dpitch:(nc - 1) * dpitch + 64]
                assert torch.equal(want, got), "ingest kernel output differs"
            emit(dict(info, leg="kernel", fmt=name, n_channels=nc, n_frames=n_frames, bytes_read=n_frames * nc * isz,
                      bytes_written=n_frames * nc * osz, ms=round(ms, 4), gbs=round(gbs, 1), d2d_copy_ms=round(ms_copy, 4),
                      d2d_copy_gbs=round(copy_gbs, 1), frac_of_copy=round(gbs / copy_gbs, 3)))
            del src, dst, rows, cp
            torch.cuda.empty_cache()


def numpy_leg(args, info, emit):
    for name, dt in (("s16", np.int16), ("f32", np.float32)):
        for nc in CHANNELS[1:]:   # one channel needs no deinterleave
            n_frames = int(args.host_gb * (1 << 30)) // (nc * np.dtype(dt).itemsize)
            frames = np.random.default_rng(1).integers(-30000, 30000, (n_frames, nc)).astype(dt)
            np.ascontiguousarray(frames[:1024].T)
            t0 = time.perf_counter()
            planar = np.ascontiguousarray(frames.T)
            s = time.perf_counter() - t0
            emit(dict(info, leg="numpy", fmt=name, n_channels=nc, n_frames=n_frames, seconds=round(s, 4),
                      gbs=round(2 * frames.nbytes / s / 1e9, 2), how="np.ascontiguousarray(frames.T), one thread"))
            del frames, planar


def e2e_leg(args, info, emit):
    import torch
    lib = _lib.load()
    rate, ns = 22050, args.streams
    n = int(args.seconds * rate)
    stride = (n + 7) // 8 * 8
    buf = torch.empty((ns, stride), dtype=torch.int16, device="cuda")
    synth.generate_on_device(synth.plan_corpus(ns, rate, args.seconds), buf.data_ptr(), stride, n, rate, device=0)
    hp = lib.same_host_alloc(ns * stride * 2)
    hi = lib.same_host_alloc(ns * n * 2)
    assert hp and hi, "pinned host allocation failed"
    planar = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_int16)), shape=(ns, stride))
    inter = np.ctypeslib.as_array(C.cast(hi, C.POINTER(C.c_int16)), shape=(n, ns))
    torch.from_numpy(planar).copy_(buf)
    torch.from_numpy(inter).copy_(buf[:, :n].t().contiguous())
    torch.cuda.synchronize()
    del buf
    torch.cuda.empty_cache()
    bounds = [int(round(i * n / args.chunks)) for i in range(args.chunks + 1)]
    rx = sb.SameReceiverBuilder.samedec(rate).build_batch(ns)

    def step(arm):
        rx.reset()
        for c in range(args.chunks):
            if arm == "planar":
                rx.submit_2d(hp, stride, bounds[c], bounds[c + 1] - bounds[c])
            else:
                rx._ck(lib.same_engine_submit_interleaved(rx.handle, C.c_void_p(hi + bounds[c] * ns * 2), 0, ns,
                                                          bounds[c + 1] - bounds[c], None))
        rx.sync()
        return rx.drain_raw()

    def canon(raw):
        """payload offsets follow the order of the device's atomics: the events with their payload bytes"""
        ev, pay = raw
        return sorted((e.stream,) + e.key() for e in sb.SameBatchReceiver.events_from_raw(ev, pay)), int((ev["kind"] == 18).sum())

    ref = {arm: canon(step(arm)) for arm in ("planar", "interleaved")}   # warm-up
    assert ref["planar"] == ref["interleaved"], "interleaved events differ from planar"
    times = {"planar": [], "interleaved": []}
    for _ in range(args.steps):
        for arm in ("planar", "interleaved"):
            l0 = rx.launch_count()
            rx.timer_start()
            got = step(arm)
            times[arm].append(rx.timer_stop())
            assert canon(got) == ref["planar"], f"{arm}: events differ"
            launches = rx.launch_count() - l0
            times.setdefault(arm + "_launches", launches)
    ms = C.c_float()
    width = (bounds[1] - bounds[0]) * 2
    rc = lib.same_h2d_probe(0, C.c_void_p(hp), stride * 2, width, ns, args.chunks, C.byref(ms))
    probe_planar = ms.value if rc == 0 else float("nan")
    rc = lib.same_h2d_probe(0, C.c_void_p(hi), width * ns, width * ns, 1, args.chunks, C.byref(ms))
    probe_inter = ms.value if rc == 0 else float("nan")
    nbytes = ns * n * 2
    for arm, probe, geom in (("planar", probe_planar, f"{args.chunks} x ({ns} rows x {width} B, pitch {stride * 2} B)"),
                             ("interleaved", probe_inter, f"{args.chunks} x (1 row x {width * ns} B)")):
        best = min(times[arm])
        emit(dict(info, leg="e2e", arm=arm, streams=ns, seconds=args.seconds, chunks=args.chunks, headers=ref["planar"][1],
                  launches_per_step=times[arm + "_launches"], ms_per_step=[round(t, 2) for t in times[arm]],
                  audio_s_per_s=round(ns * n / rate / (best * 1e-3), 1), h2d_gbs=round(nbytes / best / 1e6, 2),
                  h2d_probe_gbs=round(nbytes / probe / 1e6, 2), frac_of_h2d_probe=round(probe / best, 4),
                  probe_geometry=geom))
    lib.same_host_free(hp)
    lib.same_host_free(hi)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--gb", type=float, default=1.0, help="kernel leg: GiB of input per case")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-gb", type=float, default=0.25, help="numpy leg: GiB per block")
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--chunks", type=int, default=24)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--legs", default="kernel,e2e,numpy")
    args = ap.parse_args()
    info = card()

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    legs = args.legs.split(",")
    if "kernel" in legs:
        kernel_leg(args, info, emit)
    if "numpy" in legs:
        numpy_leg(args, info, emit)
    if "e2e" in legs:
        e2e_leg(args, info, emit)


if __name__ == "__main__":
    main()

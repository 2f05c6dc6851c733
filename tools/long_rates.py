"""Long-stream path at every input rate: ONE stream per rate (22 050, 44 100, 48 000, 96 000, 192 000 Hz), decoded by a
one-stream engine with long_stream = 1 (same_long.cu) and with long_stream = 0 (the ordinary kernels: the pipelined
kernel at 22 050 Hz, the rate-generic or wide kernel elsewhere), on two signals:
  corpus  plan_long_stream (SAME events every 10-60 minutes over the corpus noise, sigma 3663), device generator
  quiet   burst-free noise of sigma 500 (-36 dBFS), where the speculative AGC's hand-overs mostly fail to verify

Time = host clock around submit + sync of one submit from device memory (ends in a device synchronise; no host->device
copy inside), after one warm-up submit per engine configuration.  The long arm decodes --hours of audio; the ordinary
arm at most --ordinary-minutes (half of it from 88 200 Hz up), since it runs at 20-130x realtime there: the comparison
is in x realtime.  Median of --reps runs, the arms alternating within each rep.  The device name, power limit and max
SM clock are read in the same run.  One JSON line per (rate, signal, arm).
usage: python tools/long_rates.py [--hours H] [--ordinary-minutes M] [--rates R ...] [--reps N] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
    except Exception:
        import torch
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return name, power, clock


def signal(kind, rate, n):
    """n device samples (torch int16) of the signal"""
    import torch

    from sameold_b200 import synth
    buf = torch.empty(((n + 7) // 8 * 8,), dtype=torch.int16, device="cuda")
    if kind == "corpus":
        plan = synth.plan_long_stream(n / rate / 3600.0, rate)
        synth.DeviceCorpus([plan], rate).generate(buf.data_ptr(), buf.numel(), n)
    else:
        plan = synth.StreamPlan("", [], [], 0.0, 0x51 + rate)
        synth.DeviceCorpus([plan], rate, noise_sigma=500.0).generate(buf.data_ptr(), buf.numel(), n)
    torch.cuda.synchronize()
    return buf


def run_one(b, buf, n, long_stream):
    import numpy as np
    import torch
    off = np.zeros(1, np.uint64)
    warm = b.build_batch(1)
    warm.set_option("long_stream", long_stream)
    warm.submit_device(buf.data_ptr(), n, off, np.array([min(n, 1 << 18)], np.uint32))
    warm.sync()
    warm.close()
    rx = b.build_batch(1)
    rx.set_option("long_stream", long_stream)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rx.submit_device(buf.data_ptr(), n, off, np.array([n], np.uint32))
    rx.sync()
    dt = time.perf_counter() - t0
    n_events = len(rx.drain_raw()[0])
    out = {"seconds": dt, "events": n_events, "long_stream_passes": rx.get_option("long_stream_passes"),
           "long_stream_fallback_spans": rx.get_option("long_stream_fallback_spans")}
    rx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=1.0)
    ap.add_argument("--ordinary-minutes", type=float, default=10.0)
    ap.add_argument("--rates", type=int, nargs="+", default=[22050, 44100, 48000, 96000, 192000])
    ap.add_argument("--signals", nargs="+", default=["corpus", "quiet"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import sameold_b200 as sb
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    name, power, clock = device_info()
    lines = []
    for rate in args.rates:
        b = sb.SameReceiverBuilder.samedec(rate)
        n_long = int(args.hours * 3600 * rate)
        minutes = args.ordinary_minutes / (2 if rate >= 88200 else 1)
        n_ord = min(n_long, int(minutes * 60 * rate))
        for kind in args.signals:
            buf = signal(kind, rate, n_long)
            runs = {1: [], 0: []}
            for _ in range(args.reps):
                for ls, n in ((1, n_long), (0, n_ord)):
                    runs[ls].append(run_one(b, buf, n, ls))
            for ls, n in ((1, n_long), (0, n_ord)):
                rs = runs[ls]
                secs = sorted(r["seconds"] for r in rs)
                med = secs[len(secs) // 2]
                audio = n / rate
                rec = {"rate": rate, "signal": kind, "long_stream": ls, "audio_seconds": audio, "seconds_median": med,
                       "seconds_all": secs, "x_realtime_median": audio / med, "events": rs[-1]["events"],
                       "long_stream_passes": rs[-1]["long_stream_passes"],
                       "long_stream_fallback_spans": rs[-1]["long_stream_fallback_spans"],
                       "device": name, "power_limit": power, "max_sm_clock": clock}
                lines.append(json.dumps(rec))
                print(lines[-1], flush=True)
            del buf
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

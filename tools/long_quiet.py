"""Long-stream path on burst-free noise: one stream, one hour of white noise at a given level, submitted as one chunk
from device memory, through the long-stream path (same_long.cu) and with option long_stream = 0 (the ordinary
kernels).  At sigma 500 (-36 dBFS) the speculative AGC's hand-overs mostly fail to verify (DESIGN.md §4), so this is
the input that exercises the long path's verification stops; sigma 3663 is the corpus noise, where every hand-over
verifies.

Time = host clock around submit + sync (ends in a device synchronise; no host->device copy inside: the samples are
already on the device), median of --reps runs after one warm-up submit.  Each library given with --lib LABEL=PATH
runs in a process of its own (SAME_B200_LIB), the libraries alternating rep by rep; without --lib the tree's build
runs.  The device name and power limit are read in the same run.  One JSON line per (library, sigma, path).
usage: python tools/long_quiet.py [--hours H] [--sigma S ...] [--reps N] [--lib LABEL=PATH ...] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RATE = 22050


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
    except Exception:
        import torch
        name, power, clock = torch.cuda.get_device_name(0), "unknown", "unknown"
    return name, power, clock


def noise(sigma, n, seed=0x51):
    import numpy as np
    rng = np.random.Generator(np.random.Philox(key=seed + int(sigma)))
    out = np.empty(n, np.int16)
    step = 1 << 24
    for lo in range(0, n, step):
        m = min(step, n - lo)
        out[lo:lo + m] = np.clip(np.rint(rng.standard_normal(m) * sigma), -32768, 32767)
    return out


def run_one(sigma, hours, long_stream):
    """seconds for one hour-long submit, and the engine's long-path counters"""
    import numpy as np
    import torch

    import sameold_b200 as sb
    n = int(hours * 3600 * RATE)
    x = torch.from_numpy(noise(sigma, n)).cuda()
    b = sb.SameReceiverBuilder.samedec(RATE)
    off, ln = np.zeros(1, np.uint64), np.array([n], np.uint32)
    warm = b.build_batch(1)
    warm.set_option("long_stream", long_stream)
    warm.submit_device(x.data_ptr(), n, off, np.array([min(n, 1 << 18)], np.uint32))
    warm.sync()
    warm.close()
    rx = b.build_batch(1)
    rx.set_option("long_stream", long_stream)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rx.submit_device(x.data_ptr(), n, off, ln)
    rx.sync()
    dt = time.perf_counter() - t0
    rx.drain_raw()
    out = {"seconds": dt, "x_realtime": hours * 3600 / dt,
           "long_stream_passes": rx.get_option("long_stream_passes"),
           "long_stream_fallback_spans": rx.get_option("long_stream_fallback_spans")}
    rx.close()
    return out


def child(args):
    for sigma in args.sigma:
        for ls in (1, 0):
            print(json.dumps({"sigma": sigma, "long_stream": ls, **run_one(sigma, args.hours, ls)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=1.0)
    ap.add_argument("--sigma", type=float, nargs="+", default=[500.0, 3663.0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lib", action="append", default=[], help="LABEL=PATH of an in-tree build of the same ABI")
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        child(args)
        return
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", "")]
    name, power, clock = device_info()
    runs = {}
    for rep in range(args.reps):
        for label, path in libs:
            env = dict(os.environ)
            if path:
                env["SAME_B200_LIB"] = os.path.abspath(path)
            cmd = [sys.executable, os.path.abspath(__file__), "--child", "--hours", str(args.hours), "--sigma"]
            cmd += [str(s) for s in args.sigma]
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True)
            for line in r.stdout.splitlines():
                d = json.loads(line)
                runs.setdefault((label, d["sigma"], d["long_stream"]), []).append(d)
    lines = []
    for (label, sigma, ls), rs in runs.items():
        secs = sorted(r["seconds"] for r in rs)
        rec = {"lib": label, "sigma": sigma, "long_stream": ls, "hours": args.hours, "seconds_median": secs[len(secs) // 2],
               "seconds_all": secs, "x_realtime_median": args.hours * 3600 / secs[len(secs) // 2],
               "long_stream_passes": rs[-1]["long_stream_passes"],
               "long_stream_fallback_spans": rs[-1]["long_stream_fallback_spans"],
               "device": name, "power_limit": power, "max_sm_clock": clock}
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

"""Throughput of the receiver at wide input rates: 48 kHz (the rate-generic kernel, as a reference point), 96 kHz and
192 kHz (the wide kernel), for 1 .. 16384 streams, plus the CPU oracle on every host core at 192 kHz as the baseline.

Corpus: device-resident synthetic streams (DeviceCorpus, the config-3 signal model: 3 header + 3 EOM bursts, AWGN at
10 dB SNR, +-5 Hz offset) of --seconds each at the target rate, samedec configuration.  Each stream is submitted from
device memory in --chunk-seconds pieces (the state stays resident between them), so the largest point needs only one
chunk of samples on the device.  Kernel time = CUDA events around each launch (same_engine_last_timing), summed over
the chunks after one warm-up engine per rate.  Resident 32-stream blocks per SM come from the CUDA runtime's occupancy
calculator (engine option "resident_blocks_per_sm").  One JSON line per point; the device name, power limit and maximum
SM clock are read in the same run, and the library (SAME_B200_LIB, else the tree's build) is named.  --out FILE also
appends the lines to FILE.
usage: python tools/wide_rates.py [--rates R ...] [--streams N ...] [--seconds S] [--chunk-seconds C] [--cpu-streams K]
"""
import argparse
import json
import os
import subprocess
import sys

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


def kernel_name(rate):
    """the receiver kernel an engine at `rate` (samedec configuration) launches"""
    import numpy as np
    sps = np.float32(rate) / np.float32(520.83)
    ntaps, dc = int(np.floor(sps)), int(np.float32(0.38) * sps)
    return "same_rx_generic_kernel" if ntaps <= 128 and dc <= 64 else "same_rx_wide_kernel"


def run_point(rate, ns, seconds, chunk_seconds):
    import numpy as np
    import torch

    import sameold_b200 as sb
    from sameold_b200 import synth
    n = int(seconds * rate)
    cn = min(n, int(chunk_seconds * rate) // 8 * 8)
    corpus = synth.DeviceCorpus(synth.plan_corpus(ns, rate, seconds), rate)
    buf = torch.empty((ns, cn), dtype=torch.int16, device="cuda")
    rx = sb.SameReceiverBuilder.samedec(rate).build_batch(ns)
    rx.set_event_capacity(max(65536, ns * 16), max(4 << 20, ns * 2048))
    offsets = np.arange(ns, dtype=np.uint64) * cn
    resident = rx.get_option("resident_blocks_per_sm")
    kernel_ms, launches, events, som = 0.0, 0, 0, 0
    for first in range(0, n, cn):
        m = min(cn, n - first)
        corpus.generate(buf.data_ptr(), cn, m, first)
        torch.cuda.synchronize()
        rx.submit_device(buf.data_ptr(), ns * cn, offsets, np.full(ns, m, np.uint32))
        rx.sync()
        kernel_ms += rx.last_timing()[1]
        launches += 1
        for e in rx.drain():
            events += 1
            som += e.kind == 18
    audio = ns * seconds
    return {"rate_hz": rate, "streams": ns, "seconds": seconds, "launches": launches,
            "kernel_ms_per_launch": round(kernel_ms / launches, 3), "kernel_ms_total": round(kernel_ms, 3),
            "audio_s_per_s": round(audio / (kernel_ms / 1e3), 1), "samples_per_s": float(f"{audio * rate / (kernel_ms / 1e3):.4g}"),
            "events": events, "som": som, "resident_blocks_per_sm": resident}


def run_cpu(rate, ns, seconds):
    import numpy as np
    import torch

    import sameold_b200 as sb
    from oracle.pyoracle import Oracle, OracleConfig
    from sameold_b200 import synth
    n = int(seconds * rate)
    buf = torch.empty((ns, n), dtype=torch.int16, device="cuda")
    synth.DeviceCorpus(synth.plan_corpus(ns, rate, seconds), rate).generate(buf.data_ptr(), n, n)
    host = buf.cpu().numpy()
    c, o = sb.SameReceiverBuilder.samedec(rate).config(), OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(c, name))
    cores = os.cpu_count() or 1
    secs, nb, nm = Oracle.decode_batch(o, host, cores)
    return {"rate_hz": rate, "streams": ns, "seconds": seconds, "cpu_oracle_threads": cores, "wall_s": round(secs, 3),
            "audio_s_per_s": round(ns * seconds / secs, 1), "samples_per_s": float(f"{ns * seconds * rate / secs:.4g}"),
            "bursts": int(np.sum(nb)), "messages": int(np.sum(nm))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rates", type=int, nargs="+", default=[48000, 96000, 192000])
    ap.add_argument("--streams", type=int, nargs="+", default=[1, 1024, 4096, 4736, 16384])
    ap.add_argument("--seconds", type=float, default=20.0)
    ap.add_argument("--chunk-seconds", type=float, default=5.0)
    ap.add_argument("--cpu-streams", type=int, default=64, help="CPU oracle baseline at the highest rate (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "wide_rates.py measures the GPU: no CUDA device"
    name, power, clock = device_info()
    common = {"gpu": name, "power_limit": power, "max_sm_clock": clock,
              "lib": os.path.basename(os.environ.get("SAME_B200_LIB", "libsame_b200.so"))}
    lines = []
    for rate in args.rates:
        run_point(rate, 32, 0.5, 0.5)   # warm-up: module load, first launch at this geometry
        for ns in args.streams:
            rec = run_point(rate, ns, args.seconds, args.chunk_seconds)
            rec.update(common, kernel=kernel_name(rate))
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if args.cpu_streams:
        rec = run_cpu(max(args.rates), args.cpu_streams, args.seconds)
        rec.update(common, kernel="cpu_oracle")
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

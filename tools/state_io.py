"""Cost of exporting and importing stream state (same_engine_export_streams / same_engine_import_streams) on one GPU.

For 4096 and 65536 streams, after a 10 s synthetic prefix: export split into the gather+CRC kernel and the
device->host copy, import split into the host->device copy and validate+scatter, bytes per stream, with a pinned and
with a pageable host buffer.  Times are CUDA-event times the engine reports ("state_kernel_us" / "state_copy_us"),
median of several repetitions; the device name and power limit are read in the same run.
usage: python tools/state_io.py [--out FILE] [--reps N]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import sameold_b200 as sb  # noqa: E402
from sameold_b200 import _lib, synth  # noqa: E402


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
    except Exception:
        import torch
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def prefix(rx, n, seconds, rate=22050):
    plans = [synth.plan_stream(i, seconds=seconds) for i in range(64)]
    base = np.stack([synth.render_numpy(p, seconds * rate) for p in plans])
    rows = np.arange(n) % 64
    for c0 in range(0, seconds * rate, rate):
        rx.submit(np.ascontiguousarray(base[rows, c0:c0 + rate]))
        rx.sync()
        rx.drain_raw(reuse=True)


def measure(n, reps, seconds):
    lib = _lib.load()
    rx = sb.SameReceiverBuilder.samedec(22050).build_batch(n)
    prefix(rx, n, seconds)
    size = lib.same_engine_state_bytes(rx.handle, n)
    pinned_p = lib.same_host_alloc(size)
    pinned = np.ctypeslib.as_array(C.cast(pinned_p, C.POINTER(C.c_uint8)), shape=(size,))
    pageable = np.empty(size, np.uint8)
    pageable[:] = 1                                   # touch the pages before timing
    out = {"streams": n, "bytes_total": int(size), "bytes_per_stream": (size - 2224) / n}
    written = C.c_size_t()
    ids = np.arange(n, dtype=np.uint32)
    for kind, buf in (("pinned", pinned), ("pageable", pageable)):
        ek, ec, ic, ik = [], [], [], []
        for _ in range(reps):
            rx._ck(lib.same_engine_export_streams(rx.handle, None, n, buf.ctypes.data, size, C.byref(written)))
            ek.append(rx.get_option("state_kernel_us") / 1e3)
            ec.append(rx.get_option("state_copy_us") / 1e3)
            rx._ck(lib.same_engine_import_streams(rx.handle, ids.ctypes.data, n, buf.ctypes.data, size))
            ic.append(rx.get_option("state_copy_us") / 1e3)
            ik.append(rx.get_option("state_kernel_us") / 1e3)
        med = lambda v: float(np.median(v))  # noqa: E731
        out[kind] = {"export_gather_crc_ms": med(ek), "export_d2h_ms": med(ec), "import_h2d_ms": med(ic),
                     "import_validate_scatter_ms": med(ik),
                     "d2h_GBps": size / med(ec) / 1e6 if med(ec) else None,
                     "h2d_GBps": size / med(ic) / 1e6 if med(ic) else None}
    lib.same_host_free(C.c_void_p(pinned_p))
    rx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seconds", type=int, default=10)
    args = ap.parse_args()
    name, power = device_info()
    res = {"device": name, "power_limit": power, "prefix_seconds": args.seconds, "reps": args.reps,
           "runs": [measure(n, args.reps, args.seconds) for n in (4096, 65536)]}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

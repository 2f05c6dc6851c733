#!/usr/bin/env python3
"""bench.py — aggregate audio-seconds decoded per second (BASELINE.json metric) on N B200s.

A step = one pass of the receiver hot path over one batch: `streams` synthetic 60 s s16le streams per GPU at 22050 Hz
(BASELINE.md config 3: SAME bursts, AWGN 10 dB SNR, +-5 Hz offset), every stream decoded from a freshly reset receiver.
Weak scaling: every GPU gets its own `streams` streams (different seeds); no collective on the data path — NCCL is used
only for the barrier and the max-over-ranks of the measured time.

  value     device-resident inputs, CUDA-event time of K steps on the engine's own streams (reset + kernel + event read-back)
  e2e       same workload from pinned HOST memory through the C ABI (same_engine_submit_s16_2d), time-chunked so the
            host->device copy of chunk k+1 overlaps the kernel of chunk k; events copied back to the host every step
  roofline  algorithmic bytes (2 B/sample, SURVEY.md §8d) of one receiver-kernel launch / its CUDA-event duration,
            against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (C++ restatement of sameold 0.6.0, one stream per host thread) on a bounded sample of the
            same corpus — `kind: "port"` (the Rust reference cannot be built here)

  config4   (extra key of the same line) BASELINE config 4: 65 536 streams x 60 s in TOTAL (173 GB), contiguous shards
            of 65 536/N streams per rank, streamed through in 5 s time-chunks with the receiver state resident
            (strong scaling); device-resident and host-buffer numbers like `value` / `e2e`
  e2e.h2d_ceiling_gbs  bare pinned host->device copy rate of all ranks at once (no kernel): what `e2e` is bounded by

`--impl reference` times that CPU implementation alone (rank 0 only), same metric/config.
`--config 5` runs BASELINE config 5 (one 24 h stream) on one GPU and prints its own line.
`--dump-outputs DIR` writes the events of the last timed step (rank 0) as .npy files, see dump_outputs().
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RATE = 22050
METRIC = "audio_seconds_decoded_per_second"
UNIT = "audio-s/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU (config 3: 4096)")
    ap.add_argument("--seconds", type=float, default=60.0, help="stream duration")
    ap.add_argument("--e2e-chunks", type=int, default=24, help="time-chunks per step on the host-buffer path")
    ap.add_argument("--cpu-sample-streams", type=int, default=1024)
    ap.add_argument("--no-bursts", action="store_true", help="diagnostic: noise-only corpus (not a valid bench line)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the config-4 leg (65536 streams, time-chunked, sharded)")
    ap.add_argument("--config", type=int, default=3, choices=[3, 5], help="5: the single 24 h stream (own JSON line)")
    ap.add_argument("--hours", type=float, default=24.0, help="--config 5 stream length")
    ap.add_argument("--config4-streams", type=int, default=65536)
    ap.add_argument("--config4-chunk-seconds", type=float, default=5.0)
    ap.add_argument("--kernel", type=int, default=0, help="diagnostic: engine option 'kernel' (0 = measured policy)")
    ap.add_argument("--lanes-per-warp", type=int, default=0, help="diagnostic: engine option 'lanes_per_warp'")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the events the last timed step drained (rank 0) to DIR/*.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.config == 5:
        ap.error("--dump-outputs covers the config-3 step; --config 5 has no step to dump")
    return args


def workload_name(streams, seconds):
    return (f"config3: {streams} synthetic {seconds:g} s streams per GPU @22050 Hz s16le, 3 header + 3 EOM SAME bursts, "
            f"AWGN 10 dB SNR, +-5 Hz tone offset, seed 0x5A3E0000+stream_id")


class ClockSampler:
    """SM clock + throttle reasons of this rank's GPU during the timed region (B200_PROFILING.md recipe): NVML polled
    from a thread every 10 ms (no process start-up, so even a sub-second region gets samples); `nvidia-smi -lms` is the
    fallback when NVML cannot be loaded."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.thread, self.stop_flag = None, None, None, threading.Event()
        self.sm, self.max_sm, self.bits = [], None, 0
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(index)
            bus = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.bits |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass
            self.stop_flag.wait(0.01)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            n = self.nvml
            masks = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
            reasons = [name for name, m in zip(self.NAMES, masks) if self.bits & m]
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_sm,
                    "samples": len(self.sm), "reasons": reasons, "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) >= 8 and r[4 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons, "source": "nvidia-smi"}


def oracle_config_from(cfg):
    from oracle.pyoracle import OracleConfig
    o = OracleConfig()
    for name, _ in OracleConfig._fields_:
        setattr(o, name, getattr(cfg, name))
    return o


def cpu_baseline(host_samples, cfg, cores):
    """Oracle on the host cores: one receiver per stream, `cores` threads (BASELINE.md §4).  Best of 2."""
    from oracle import Oracle
    ocfg = oracle_config_from(cfg)
    best = None
    for _ in range(2):
        secs, nb, nm = Oracle.decode_batch(ocfg, host_samples, cores)
        best = secs if best is None else min(best, secs)
    audio = host_samples.shape[0] * host_samples.shape[1] / RATE
    return audio / best, best, int(nb.sum()), int(nm.sum())


def _cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if part:
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_host_cpus(device, local_rank, local_world):
    """Pin this process — and with it the first-touch placement of its pinned sample pool, allocated afterwards — to
    host cores next to its GPU, so that with one rank per GPU the host->device copies of different ranks do not cross
    the socket interconnect and the ranks' host threads do not migrate onto each other.  In order: the NUMA node sysfs
    reports for the GPU; the CPU affinity NVML reports for it (what `nvidia-smi topo -m` prints); an even split of
    the allowed cores per local rank (single-node VMs report neither).  Returns a description for the bench line."""
    allowed = os.sched_getaffinity(0)
    try:
        import torch
        props = torch.cuda.get_device_properties(device)
        bus = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node >= 0:
            cpus = _cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read()) & allowed
            if cpus and len(cpus) < len(allowed):
                os.sched_setaffinity(0, cpus)
                return {"how": "sysfs numa_node", "node": node, "cpus": len(cpus)}
    except Exception:
        pass
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(device)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1} & allowed
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return {"how": "nvml cpu affinity", "node": None, "cpus": len(cpus)}
    except Exception:
        pass
    try:
        cores = sorted(allowed)
        per = max(1, len(cores) // max(1, local_world))
        mine = set(cores[local_rank * per:(local_rank + 1) * per]) or set(cores)
        os.sched_setaffinity(0, mine)
        return {"how": "even split of allowed cores (no NUMA information on this box)", "node": None, "cpus": len(mine)}
    except Exception:
        return {"how": "unbound", "node": None, "cpus": len(allowed)}


def device_for_rank(local_rank, local_world, n_devices):
    """Which GPU a rank drives when the box has more GPUs than the job has ranks: the ranks are striped over the device
    index range (8 GPUs: 0, 4, 1, 5, 2, 6, 3, 7) instead of packed into the first N.  Measured on this pod's 8-GPU
    boxes (profiles/README.md, round 2): GPUs 0-3 share one host path that sustains ~115 GB/s of pinned host->device
    copies in total (29 GB/s each when all four copy, 55 GB/s each for any two), GPUs 4-7 another; `nvidia-smi topo`
    and sysfs expose nothing (one NUMA node), so the order is a static spread, not a lookup."""
    if local_world <= 1 or n_devices <= local_world:
        return local_rank
    half = n_devices // 2
    order = [i // 2 + (i % 2) * half for i in range(2 * half)] + list(range(2 * half, n_devices))
    return order[local_rank]


def kernel_source_sha16():
    """Hash of the receiver-kernel sources: ties profiles/rx_kernel_traffic.json (an ncu capture) to the code it was
    taken from, so a stale capture is dropped instead of silently reported."""
    import hashlib
    h = hashlib.sha256()
    for f in ("same_kernels.cu", "same_fast.cuh", "same_lane.cuh", "same_transport.cuh", "same_params.h"):
        with open(os.path.join(ROOT, "sameold_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def profiled_traffic(ns, seconds):
    """(dram bytes per launch from the committed ncu capture or None, note)."""
    tpath = os.path.join(ROOT, "profiles", "rx_kernel_traffic.json")
    try:
        tj = json.load(open(tpath))
    except Exception:
        return None, "no ncu capture committed"
    if tj.get("streams") != ns or abs(tj.get("seconds", 0) - seconds) > 1e-9:
        return None, "ncu capture is for another workload"
    if tj.get("kernel_src_sha16") != kernel_source_sha16():
        return None, f"ncu capture of {tj.get('captured', '?')} predates the current kernel sources (stale): dropped"
    return tj.get("dram_bytes_per_launch"), f"ncu --set full capture of {tj.get('captured', '?')} ({tj.get('report', '')})"


DUMP_MAX_BYTES = 64 * 10 ** 6


def canonical_events(evs, pay):
    """One drain's same_event records and payload, with every event's payload bytes laid out in event order and
    `data_offset` pointing there.  Where a device drain places a payload in its arena depends on which warp wrote
    first, so only this form is comparable from run to run.  link.Burst (kind 3) payloads are stored up to
    SAME_BURST_CAP = 1024 bytes; `data_len` keeps the true length."""
    e = np.array(evs, copy=True)
    stored = np.where(e["kind"] == 3, np.minimum(e["data_len"], 1024), e["data_len"]).astype(np.int64)
    start = np.cumsum(stored) - stored
    idx = np.repeat(e["data_offset"].astype(np.int64) - start, stored) + np.arange(int(stored.sum()))
    e["data_offset"] = start
    return e, np.asarray(pay)[idx]


def dump_outputs(dirname, evs, pay, n_streams, max_bytes=DUMP_MAX_BYTES):
    """Write one drain in canonical_events form: DIR/event_<field>.npy for each same_event field (float64: every value
    is an integer below 2^53) and DIR/payload.npy (the payload bytes, float32), plus DIR/streams.npy, the streams
    included.  When all streams do not fit in `max_bytes`, the longest prefix that fits of a fixed seeded permutation
    of the streams is written, in stream order, so the same events always give the same files.  Returns
    (streams written, events written)."""
    evs, pay = canonical_events(evs, pay)
    fields = evs.dtype.names
    stored = np.diff(np.append(evs["data_offset"].astype(np.int64), pay.size))
    per_stream = np.bincount(evs["stream"], weights=8 * len(fields) + 4 * stored, minlength=n_streams) + 8
    order = np.random.default_rng(0x5A3E).permutation(n_streams)
    budget = max_bytes - 4096 * (len(fields) + 2)                 # room for the .npy headers
    keep = np.sort(order[:int((np.cumsum(per_stream[order]) <= budget).sum())])
    evs, pay = canonical_events(evs[np.isin(evs["stream"], keep)], pay)
    os.makedirs(dirname, exist_ok=True)
    for f in fields:
        np.save(os.path.join(dirname, f"event_{f}.npy"), evs[f].astype(np.float64))
    np.save(os.path.join(dirname, "payload.npy"), pay.astype(np.float32))
    np.save(os.path.join(dirname, "streams.npy"), keep.astype(np.float64))
    return int(keep.size), int(evs.size)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    n_samples = int(args.seconds * RATE)
    cfgname = {"workload": workload_name(args.streams, args.seconds), "streams_per_gpu": args.streams,
               "seconds": args.seconds, "rate_hz": RATE, "receiver_config": "samedec (main.rs:29-37)",
               "l2": "inputs_exceed_l2"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        return run_reference(args, cfgname, n_samples)

    import torch
    import torch.distributed as dist
    import sameold_b200 as sb
    from sameold_b200 import synth, _lib

    all_cores = os.sched_getaffinity(0)
    device = device_for_rank(local_rank, local_world, torch.cuda.device_count())
    torch.cuda.set_device(device)
    binding = bind_host_cpus(device, local_rank, local_world) if world > 1 else {"how": "single rank: unbound", "node": None,
                                                                                  "cpus": len(all_cores)}
    binding["rank_to_device"] = [device_for_rank(r, local_world, torch.cuda.device_count()) for r in range(local_world)]
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    comm = {"world": world, "rank": rank, "local_rank": device, "barrier": barrier, "max": max_over_ranks,
            "sum": sum_over_ranks}
    if args.config == 5:
        return run_config5(args, comm)

    # ---- synthetic corpus, resident in HBM ----
    ns = args.streams
    stride = (n_samples + 7) // 8 * 8
    buf = torch.empty((ns, stride), dtype=torch.int16, device="cuda")
    plans = synth.plan_corpus(ns, RATE, args.seconds, first_stream=rank * ns)
    if args.no_bursts:
        for pl in plans:
            pl.burst_starts, pl.burst_payloads = [], []
    synth.generate_on_device(plans, buf.data_ptr(), stride, n_samples, RATE, device=device)
    offsets = np.arange(ns, dtype=np.uint64) * np.uint64(stride)
    lengths = np.full(ns, n_samples, np.uint32)

    builder = sb.SameReceiverBuilder.samedec(RATE)
    rx = builder.build_batch(ns, device=device)
    if args.kernel:
        rx.set_option("kernel", args.kernel)
    if args.lanes_per_warp:
        rx.set_option("lanes_per_warp", args.lanes_per_warp)
    kernel_names = {1: "same_rx_generic_kernel", 2: "same_rx_fast_kernel", 3: "same_rx_pipe_kernel", 4: "same_rx_ws_kernel",
                    5: "same_frontend_kernel + same_rx_fast_kernel<tile-fed>", 6: "same_rx_la_kernel"}
    kernel_name = kernel_names.get(rx.get_option("kernel_selected"), "same_rx_kernel")
    audio_per_step = ns * n_samples / RATE

    def step_device():
        rx.reset()
        rx.submit_device(buf.data_ptr(), ns * stride, offsets, lengths)
        rx.sync()
        return rx.drain_raw(reuse=True)

    # correctness guard inside the bench: every step must decode the corpus (no skipped work)
    n_headers = None
    for _ in range(args.warmup):
        evs, _pay = step_device()
        n_headers, n_events = int((evs["kind"] == 18).sum()), int(evs.size)

    sampler = ClockSampler(device)
    launches0 = rx.launch_count()
    kernel_ms = []
    barrier()
    sampler.start()
    rx.timer_start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        evs, _pay = step_device()
        kernel_ms.append(rx.last_timing()[1])
    dev_ms = rx.timer_stop()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    launches = rx.launch_count() - launches0
    dev_ms = max_over_ranks(dev_ms)
    value = audio_per_step * args.steps * world / (dev_ms * 1e-3)
    if n_headers is None:       # no warm-up: the last timed step sets the reference counts
        n_headers, n_events = int((evs["kind"] == 18).sum()), int(evs.size)
    assert int((evs["kind"] == 18).sum()) == n_headers and (n_headers > 0 or args.no_bursts), "bench step lost its work"
    # drain_raw(reuse=True) hands out views that the e2e leg's drains overwrite
    last_step = (evs.copy(), _pay.copy()) if args.dump_outputs and rank == 0 else None
    if args.seconds >= 60.0 and not args.no_bursts:
        assert n_headers >= int(0.9 * ns), "corpus not decoded"

    # ---- roofline of the receiver kernel ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    k_ms = statistics.mean(kernel_ms)
    achieved = (2.0 * ns * n_samples) / (k_ms * 1e-3) / 1e9
    traffic, traffic_note = profiled_traffic(ns, args.seconds)
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 5), "traffic": traffic, "traffic_source": traffic_note,
                "peak_source": peak_src, "kernel_ms_per_launch": round(k_ms, 3),
                "algorithmic_bytes_per_launch": 2 * ns * n_samples,
                "note": "fused per-lane receiver loop is issue/latency-bound, not HBM-bound (DESIGN.md §5); the HBM-bound "
                        "feed-forward kernel (same_frontend_kernel) is measured in profiles/"}

    # ---- e2e: host buffers through the C ABI, H2D + event D2H inside the timed region ----
    e2e = None
    host_np = None
    lib = _lib.load()
    import ctypes as C
    if not args.no_e2e:
        nbytes = ns * stride * 2
        hptr = lib.same_host_alloc(nbytes)
        if not hptr:
            raise RuntimeError("pinned host allocation failed")
        host_np = np.ctypeslib.as_array(C.cast(hptr, C.POINTER(C.c_int16)), shape=(ns, stride))
        # same corpus, now in pinned host memory (copied out once, untimed)
        host_t = torch.from_numpy(host_np)
        host_t.copy_(buf)
        torch.cuda.synchronize()
        nchunk = max(1, args.e2e_chunks)
        bounds = [int(round(i * n_samples / nchunk)) for i in range(nchunk + 1)]
        d2h_bytes = []

        def step_host():
            rx.reset()
            for c in range(nchunk):
                rx.submit_2d(hptr, stride, bounds[c], bounds[c + 1] - bounds[c])
            rx.sync()
            return rx.drain_raw(reuse=True)

        for _ in range(max(1, args.warmup - 1)):
            ev, pay = step_host()
        assert int((ev["kind"] == 18).sum()) == n_headers, "chunked host path decodes differently"
        barrier()
        rx.timer_start()
        for _ in range(args.steps):
            ev, pay = step_host()
            d2h_bytes.append(48 * int(ev.size) + int(pay.size) + 8 * nchunk)
        e2e_ms = rx.timer_stop()
        barrier()
        e2e_ms = max_over_ranks(e2e_ms)
        # the ceiling: the same bytes in the same strided chunks, every rank at once, no kernel
        ms = C.c_float()
        barrier()
        width = (bounds[1] - bounds[0]) * 2
        rc = lib.same_h2d_probe(device, C.c_void_p(hptr), stride * 2, width, ns, nchunk, C.byref(ms))
        barrier()
        probe_ms = max_over_ranks(ms.value if rc == 0 else float("nan"))
        ceiling_gbs = world * ns * width * nchunk / (probe_ms * 1e-3) / 1e9
        e2e_gbs = world * ns * n_samples * 2 * args.steps / (e2e_ms * 1e-3) / 1e9
        e2e = {"value": round(audio_per_step * args.steps * world / (e2e_ms * 1e-3), 1), "unit": UNIT,
               "h2d_bytes_per_step": int(ns * n_samples * 2 + nchunk * ns * 12) * world,
               "d2h_bytes_per_step": int(sum_over_ranks(statistics.mean(d2h_bytes))), "ms_per_step": round(e2e_ms / args.steps, 3),
               "chunks_per_step": nchunk, "api": "same_engine_submit_s16_2d + sync + drain_events (pinned host buffer)",
               "h2d_gbs": round(e2e_gbs, 2), "h2d_ceiling_gbs": round(ceiling_gbs, 2),
               "frac_of_h2d_ceiling": round(e2e_gbs / ceiling_gbs, 4),
               "h2d_ceiling_how": f"same_h2d_probe: {nchunk} strided copies of {ns} rows x {width} B per rank from the same pinned "
                                  f"buffer, all {world} ranks at once, no kernel, max over ranks",
               "host_binding": binding}

    # ---- CPU baseline (rank 0's host cores; the other ranks wait) ----
    cpu = None
    if not args.no_cpu:
        if rank == 0:
            k = min(args.cpu_sample_streams, ns)
            sample = buf[:k, :n_samples].cpu().numpy()
            mine = os.sched_getaffinity(0)
            os.sched_setaffinity(0, all_cores)        # the baseline gets every host core (the other ranks wait at the barrier)
            cores = len(all_cores)
            v, secs, nb, nm = cpu_baseline(sample, builder.config(), cores)
            os.sched_setaffinity(0, mine)
            cpu = {"value": round(v, 1), "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"first {k} streams x {args.seconds:g} s of this workload, one receiver per stream, {cores} threads, best of 2 ({secs:.2f} s)",
                   "what": "oracle/ C++ restatement of sameold 0.6.0 (link + transport layers), g++ -O2 -ffp-contract=off; the Rust crate cannot be built here"}
            del sample
        barrier()

    # ---- config 4: 65 536 streams in total, sharded over the ranks, time-chunked ----
    del buf
    if host_np is not None:
        del host_np, host_t
        lib.same_host_free(hptr)
    del rx
    torch.cuda.empty_cache()
    config4 = None
    if not args.no_config4 and not args.no_bursts:
        try:
            config4 = run_config4(args, comm, peak)
        except Exception as e:  # the main line must survive a failure of the extra leg
            config4 = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfgname,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "wall_ms_per_step": round(wall_ms / args.steps, 3), "events_per_step": n_events,
            "headers_decoded_per_step": n_headers, "realtime_factor_per_gpu": round(value / world, 1),
            "config4": config4,
        }
        if last_step is not None:
            k, nev = dump_outputs(args.dump_outputs, *last_step, ns)
            print(f"dumped {nev} events of {k} streams to {args.dump_outputs}", file=sys.stderr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_config4(args, comm, peak):
    """BASELINE config 4: `config4_streams` (65 536) synthetic 60 s streams in TOTAL; rank r owns the contiguous shard
    [r*S/N, (r+1)*S/N) (one engine, one CUDA stream pair); the 173 GB of samples do not fit one GPU, so every rank
    streams its shard through in `chunk_seconds` time-chunks with the receiver state resident (chunked == whole,
    receiver.rs:233-274).  STRONG scaling: the total is fixed.  Two timings, both summed over the chunks and taken as
    the max over ranks:
      value  each chunk generated on the device (untimed), then submit + sync + drain timed with CUDA events
      e2e    each chunk staged in pinned host memory (untimed), then submit_s16_2d in 4 column slices (copy of slice
             k+1 overlaps the kernel of slice k) + sync + drain, timed with CUDA events"""
    import ctypes as C
    import torch
    import sameold_b200 as sb
    from sameold_b200 import synth, _lib
    world, rank, local_rank = comm["world"], comm["rank"], comm["local_rank"]
    total = args.config4_streams
    first, last = total * rank // world, total * (rank + 1) // world
    ns = last - first
    secs = 60.0
    cn = int(args.config4_chunk_seconds * RATE) // 8 * 8
    n = int(secs * RATE)
    nchunks = (n + cn - 1) // cn
    plans = synth.plan_corpus(ns, RATE, secs, first_stream=first)
    corpus = synth.DeviceCorpus(plans, RATE, device=local_rank)
    buf = torch.empty((ns, cn), dtype=torch.int16, device="cuda")
    rx = sb.SameReceiverBuilder.samedec(RATE).build_batch(ns, device=local_rank)
    kernel = rx.get_option("kernel_selected")
    offsets = np.arange(ns, dtype=np.uint64) * np.uint64(cn)
    lib = _lib.load()

    def pass_device():
        rx.reset()
        ms_sum, k_sum, headers = 0.0, 0.0, 0
        for c in range(nchunks):
            w = min(cn, n - c * cn)
            corpus.generate(buf.data_ptr(), cn, w, first_sample=c * cn)
            lengths = np.full(ns, w, np.uint32)
            rx.timer_start()
            rx.submit_device(buf.data_ptr(), ns * cn, offsets, lengths)
            rx.sync()
            ev, _ = rx.drain_raw(reuse=True)
            ms_sum += rx.timer_stop()
            k_sum += rx.last_timing()[1]
            headers += int((ev["kind"] == 18).sum())
        return ms_sum, k_sum, headers

    pass_device()                                  # warm-up pass (also warms the generator)
    comm["barrier"]()
    launches0 = rx.launch_count()
    dev_ms, k_ms, headers = pass_device()
    launches = rx.launch_count() - launches0
    comm["barrier"]()
    dev_ms_max = comm["max"](dev_ms)
    k_ms_max = comm["max"](k_ms)
    headers_all = int(comm["sum"](headers))
    assert headers_all >= int(0.95 * total), f"config 4 corpus not decoded: {headers_all} headers of {total}"
    audio = total * secs
    out = {"workload": f"config4: {total} synthetic 60 s streams in total @22050 Hz s16le (173 GB), contiguous shards of "
                       f"{total}//{world} streams per GPU, {nchunks} time-chunks of {cn / RATE:g} s, state resident; same "
                       f"generator as config 3 (seed 0x5A3E0000+stream_id)",
           "streams_total": total, "streams_per_gpu": ns, "chunk_seconds": cn / RATE, "chunks": nchunks,
           "scaling": "strong", "value": round(audio / (dev_ms_max * 1e-3), 1), "unit": UNIT,
           "ms_total": round(dev_ms_max, 2), "kernel_ms_total": round(k_ms_max, 2), "kernel": kernel,
           "roofline_frac": round(2.0 * ns * n / (k_ms * 1e-3) / 1e9 / peak, 5),
           "headers_decoded": headers_all, "gpu_launches": int(launches)}
    if not args.no_e2e:
        hptr = lib.same_host_alloc(ns * cn * 2)
        if not hptr:
            raise RuntimeError("pinned host allocation failed")
        try:
            host_t = torch.from_numpy(np.ctypeslib.as_array(C.cast(hptr, C.POINTER(C.c_int16)), shape=(ns, cn)))
            nsl = 4
            rx.reset()
            e2e_ms, headers, d2h = 0.0, 0, 0
            for c in range(nchunks):
                w = min(cn, n - c * cn)
                corpus.generate(buf.data_ptr(), cn, w, first_sample=c * cn)
                host_t.copy_(buf)
                torch.cuda.synchronize()
                cuts = [int(round(i * w / nsl)) for i in range(nsl + 1)]
                rx.timer_start()
                for i in range(nsl):
                    rx.submit_2d(hptr, cn, cuts[i], cuts[i + 1] - cuts[i])
                rx.sync()
                ev, pay = rx.drain_raw(reuse=True)
                e2e_ms += rx.timer_stop()
                headers += int((ev["kind"] == 18).sum())
                d2h += 48 * int(ev.size) + int(pay.size)
            comm["barrier"]()
            e2e_max = comm["max"](e2e_ms)
            assert int(comm["sum"](headers)) == headers_all, "config 4 host path decodes differently"
            out["e2e"] = {"value": round(audio / (e2e_max * 1e-3), 1), "unit": UNIT, "ms_total": round(e2e_max, 2),
                          "h2d_bytes_per_step": int(total * n * 2), "d2h_bytes_per_step": int(comm["sum"](d2h)),
                          "h2d_gbs": round(total * n * 2 / (e2e_max * 1e-3) / 1e9, 2),
                          "api": f"same_engine_submit_s16_2d x {nsl} per chunk + sync + drain_events"}
        finally:
            del host_t
            lib.same_host_free(hptr)
    del rx, buf
    torch.cuda.empty_cache()
    return out


def run_config5(args, comm):
    """BASELINE config 5: ONE continuous stream of `--hours` (24) hours, a SAME event every U(10,60) minutes, decoded by a
    one-stream engine in 10-minute chunks from device memory.  A single stream is strictly sequential
    (receiver.rs:243): one lane of one warp — the number is the single-stream realtime factor (replicas only)."""
    import torch
    import sameold_b200 as sb
    from sameold_b200 import synth
    if comm["rank"] != 0:
        return 0
    n = int(args.hours * 3600 * RATE)
    plan = synth.plan_long_stream(args.hours, RATE)
    buf = torch.empty(((n + 7) // 8 * 8,), dtype=torch.int16, device="cuda")
    synth.DeviceCorpus([plan], RATE, device=comm["local_rank"]).generate(buf.data_ptr(), buf.numel(), n)
    rx = sb.SameReceiverBuilder.samedec(RATE).build_batch(1, device=comm["local_rank"])
    if args.kernel:
        rx.set_option("kernel", args.kernel)
    step = 600 * RATE
    zero = np.zeros(1, np.uint64)
    sampler = ClockSampler(comm["local_rank"])

    def one_pass():
        rx.reset()
        msgs, k_ms = 0, 0.0
        rx.timer_start()
        for lo in range(0, n, step):
            k = min(step, n - lo)
            rx.submit_device(buf.data_ptr() + 2 * lo, k, zero, np.array([k], np.uint32))
            rx.sync()
            ev, _ = rx.drain_raw(reuse=True)
            msgs += int(((ev["kind"] == 18) | (ev["kind"] == 19)).sum())
            k_ms += rx.last_timing()[1]
        return rx.timer_stop(), k_ms, msgs

    sampler.start()
    ms, k_ms, msgs = one_pass()
    clocks = sampler.stop()
    cpu = None
    if not args.no_cpu:
        from oracle import Oracle
        sample = buf[: min(n, 3600 * RATE)].cpu().numpy()
        o = Oracle(oracle_config_from(sb.SameReceiverBuilder.samedec(RATE).config()))
        t0 = time.perf_counter()
        o.process_s16(sample)
        secs = time.perf_counter() - t0
        cpu = {"value": round(sample.size / RATE / secs, 1), "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"first {sample.size / RATE / 3600:g} h of this stream on one host core ({secs:.2f} s)"}
    line = {"metric": METRIC, "value": round(n / RATE / (ms * 1e-3), 1), "unit": UNIT, "n_gpus": 1, "steps": 1, "warmup": 0,
            "ms_per_step": round(ms, 1), "higher_is_better": True, "scaling": "replicas only (a single stream does not shard)",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config5: one continuous {args.hours:g} h stream @22050 Hz s16le ({n} samples), "
                                   f"{len(plan.burst_starts)} bursts (a SAME event every U(10,60) min), AWGN 10 dB SNR; "
                                   f"one-stream engine, 10-minute chunks from device memory", "hours": args.hours},
            "kernel_ms_total": round(k_ms, 1), "messages_decoded": msgs, "events_planned": len(plan.burst_starts) // 6,
            "realtime_factor_single_stream": round(n / RATE / (ms * 1e-3), 1), "cpu_baseline": cpu, "clocks": clocks,
            "gpu_launches": int(rx.launch_count())}
    print(json.dumps(line))
    return 0


def run_reference(args, cfgname, n_samples):
    """The reference's CPU implementation of the path (oracle port) on all host threads, on the SAME config (`streams`
    streams x `seconds`); the corpus comes from the CPU generator in oracle/ (same signal model as the device
    generator), so this arm loads no GPU code at all.  The C++ restatement of sameold 0.6.0 stands in for the Rust
    crate, which cannot be built here (no cargo/rustc, crates not vendored)."""
    from oracle import decode_batch_events, synth_cpu
    from oracle.pyoracle import default_config
    from sameold_b200 import synth          # pure-Python stream plans only; the native library is not loaded
    cores = os.cpu_count() or 1
    k = args.streams
    plans = synth.plan_corpus(k, RATE, args.seconds, first_stream=0)
    t0 = time.perf_counter()
    sample = synth_cpu(plans, n_samples, RATE, cores)
    gen_s = time.perf_counter() - t0
    ocfg = default_config(RATE, samedec=True)
    audio = k * n_samples / RATE
    for _ in range(args.warmup):
        decode_batch_events(ocfg, sample, cores)
    t0 = time.perf_counter()
    secs_total, n_som = 0.0, 0
    for _ in range(args.steps):
        ev, _pay, secs = decode_batch_events(ocfg, sample, cores)
        secs_total += secs
        n_som = int((ev["kind"] == 18).sum())
    wall = time.perf_counter() - t0
    if args.dump_outputs:
        k_dumped, nev = dump_outputs(args.dump_outputs, ev, _pay, k)
        print(f"dumped {nev} events of {k_dumped} streams to {args.dump_outputs}", file=sys.stderr)
    assert args.seconds < 60.0 or n_som >= int(0.9 * k), "reference arm did not decode its corpus"
    value = audio * args.steps / secs_total
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(secs_total / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfgname,
        "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"all {k} streams x {args.seconds:g} s per step (CPU generator oracle/synth_cpu.hpp, "
                                   f"{gen_s:.1f} s untimed), one receiver per stream, {cores} threads"},
        "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": round(wall, 2), "headers_decoded_per_step": n_som,
        "native_so_loaded": sorted({os.path.relpath(l.split()[-1], ROOT) for l in open("/proc/self/maps")
                                    if l.rstrip().endswith(".so") and l.split()[-1].startswith(ROOT)}),
    }
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it
    sys.exit(main())

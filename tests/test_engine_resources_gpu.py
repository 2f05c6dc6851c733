"""GPU tests of what an engine owns: destroying an engine gives back every byte of device memory it allocated, the
buffers it allocates on first use included, and an allocation that fails leaves the engine as it was."""
import ctypes as C
import os

import numpy as np
import pytest

import sameold_b200 as sb
from oracle import Oracle, load_golden_recording
from oracle.pyoracle import OracleConfig
from sameold_b200 import _lib

pytestmark = pytest.mark.gpu

NAMES = ["long_message", "npt", "two_and_two"]
SAME_ERR_CUDA = 4
MiB = 1 << 20


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


def _process_device_bytes():
    """Device memory of this process over all GPUs, as NVML accounts it per process: other users of a shared GPU do
    not move this figure, as they move the device-wide free memory."""
    pynvml = pytest.importorskip("pynvml")
    pynvml.nvmlInit()
    try:
        used = None
        for i in range(pynvml.nvmlDeviceGetCount()):
            for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                if p.pid == os.getpid() and p.usedGpuMemory is not None:
                    used = (used or 0) + p.usedGpuMemory
    finally:
        pynvml.nvmlShutdown()
    if used is None:
        pytest.skip("NVML reports no memory figure for this process")
    return used


def _engine_cycle(b, noise):
    """Two engines through every path that allocates on first use, then destroyed."""
    ns, n = noise.shape
    rx = b.build_batch(ns)
    rx.submit_2d(noise.ctypes.data, n, 0, n)                   # sample buffer
    rx.sync()
    rx.drain()
    rx.enable_soft_trace(256)                                  # trace buffer
    rx.set_option("kernel", 5)                                 # split pipeline: tile buffer
    rx.process([noise[s] for s in range(ns)])
    rx.set_option("kernel", 0)
    rx.reset(list(range(1, ns, 3)))                            # id list
    rx.import_streams(rx.export_streams(list(range(0, ns, 2))), list(range(0, ns, 2)))   # record staging
    snap = rx.snapshot()                                       # snapshot
    rx.restore(snap)
    rx.free_snapshot(snap)
    rx.set_event_capacity(ns * 128, ns * 8192)                 # event arenas, reallocated
    rx.process([noise[s] for s in range(ns)])
    rx.close()

    one = b.build_batch(1)
    one.process([np.tile(noise[0], 8)])                        # long-stream scratch buffers
    assert one.get_option("long_stream_passes") >= 1
    one.close()

    lib = _lib.load()
    ms = C.c_float()
    assert lib.same_h2d_probe(0, C.c_void_p(noise.ctypes.data), n * 2, n * 2, ns, 2, C.byref(ms)) == 0


def test_destroy_returns_every_lazily_allocated_buffer():
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    noise = np.random.default_rng(7).integers(-4000, 4000, size=(4096, 11025), dtype=np.int16)
    _engine_cycle(b, noise)   # the first cycle also loads the kernels and sizes the context
    level = _process_device_bytes()
    for cycle in range(3):
        _engine_cycle(b, noise)
        now = _process_device_bytes()
        assert now <= level + 4 * MiB, f"cycle {cycle + 2}: {(now - level) / MiB:.1f} MiB more than after the first cycle"


def test_failed_event_capacity_leaves_the_engine_working():
    """An arena size that cudaMalloc refuses is an error, and the engine keeps its old arenas: it still decodes the
    golden recordings bit-exactly, and the failed allocation is not reported by a later call."""
    _torch()
    b = sb.SameReceiverBuilder.samedec(22050)
    recs = [load_golden_recording(n) for n in NAMES]
    rx = b.build_batch(3)
    for max_events, max_payload in ((1 << 40, 1 << 20), (1 << 16, 1 << 50)):   # the first or the last of the arenas fails
        with pytest.raises(sb.SameEngineError) as err:
            rx.set_event_capacity(max_events, max_payload)
        assert err.value.code == SAME_ERR_CUDA
    evs = rx.process(recs)
    for s, rec in enumerate(recs):
        o = Oracle(ocfg(b))
        o.process_s16(rec)
        assert keys(evs[s]) == keys(o.events()), NAMES[s]
    assert sum(len(e) for e in evs) > 20

"""bench.py on the GPU: --dump-outputs writes exactly the events the timed path drained in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import sameold_b200 as sb
from oracle import BATCH_EVENT_DTYPE, Oracle
from sameold_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_equal_the_oracle_on_the_bench_corpus(tmp_path):
    """The product arm without warm-up, then the oracle on the same device-generated corpus: the dumped events and
    payload are its events, field for field.  A bench step starts from reset() receivers, whose AGC gain is 1.0
    (agc.rs:61) rather than a new receiver's, so the oracle receivers are reset first as well."""
    import torch
    assert torch.cuda.is_available()
    ns, secs = 40, 30.0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "0", "--streams", str(ns),
                        "--seconds", str(secs), "--no-cpu", "--no-e2e", "--no-config4", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 0
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    n = int(secs * bench.RATE)
    stride = (n + 7) // 8 * 8
    buf = torch.empty((ns, stride), dtype=torch.int16, device="cuda")
    synth.generate_on_device(synth.plan_corpus(ns, bench.RATE, secs, first_stream=0), buf.data_ptr(), stride, n, bench.RATE)
    host = buf.cpu().numpy()[:, :n]
    cfg = bench.oracle_config_from(sb.SameReceiverBuilder.samedec(bench.RATE).config())
    rows, blobs, off = [], [], 0
    for s in range(ns):
        o = Oracle(cfg)
        o.reset()
        o.process_s16(host[s])
        for i, e in enumerate(o.events()):
            rows.append((s, i, e.sample, e.symbol_count, e.kind, e.err, off, len(e.data), e.parity_errors, e.voting_bytes, 0))
            blobs.append(e.data[:1024] if e.kind == 3 else e.data)
            off += len(blobs[-1])
    ev, pay = bench.canonical_events(np.array(rows, BATCH_EVENT_DTYPE), np.frombuffer(b"".join(blobs), np.uint8))
    assert (ev["kind"] == 18).sum() >= ns // 2
    assert np.array_equal(got["streams"], np.arange(ns))
    for f in ev.dtype.names:
        assert np.array_equal(got["event_" + f], ev[f].astype(np.float64)), f
    assert np.array_equal(got["payload"], pay.astype(np.float32))

"""bench.py contract checks that need no GPU: the reference arm (CPU oracle port) prints the contract's JSON line, and
the product arm fails loudly when there is no GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--streams", "4", "--seconds", "12")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["metric"] == "audio_seconds_decoded_per_second" and line["unit"] == "audio-s/s"
    assert line["steps"] == 2 and line["warmup"] == 1 and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]
    # the reference arm runs the CPU port only: none of the product's native code is loaded
    assert line["native_so_loaded"] == ["oracle/_build/liboracle.so"], line["native_so_loaded"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0", "--streams", "2", "--seconds", "5"], capture_output=True, text=True, timeout=300,
                       cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_dumps_the_last_steps_events(tmp_path):
    """--dump-outputs: the events of the timed path's last step, canonical and in float32/float64, the same files from
    run to run; --warmup 0 is a valid setting."""
    args = ["--impl", "reference", "--steps", "2", "--warmup", "0", "--streams", "5", "--seconds", "30"]
    for d in ("a", "b"):
        r = _run(*args, "--dump-outputs", str(tmp_path / d))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    import bench
    from oracle import decode_batch_events, synth_cpu
    from oracle.pyoracle import default_config
    from sameold_b200 import synth
    x = synth_cpu(synth.plan_corpus(5, 22050, 30.0, first_stream=0), 30 * 22050, 22050, 2)
    ev, pay = bench.canonical_events(*decode_batch_events(default_config(22050, True), x, 2)[:2])
    assert np.array_equal(a["streams"], np.arange(5)) and (ev["kind"] == 18).sum() >= 4
    for f in ev.dtype.names:
        assert np.array_equal(a["event_" + f], ev[f].astype(np.float64)), f
    assert np.array_equal(a["payload"], pay.astype(np.float32))


def test_dump_outputs_keeps_to_the_size_limit(tmp_path):
    """A drain too large for the limit is written for a fixed sample of whole streams, in stream order, with the
    payload of exactly those events."""
    import bench
    from oracle import BATCH_EVENT_DTYPE
    rng = np.random.default_rng(3)
    ns, per = 200, 7
    ev = np.zeros(ns * per, BATCH_EVENT_DTYPE)
    ev["stream"] = np.repeat(np.arange(ns), per)
    ev["seq"] = np.tile(np.arange(per), ns)
    ev["kind"] = np.tile([1, 2, 3, 17, 18, 19, 0], ns)
    ev["data_len"] = np.where(ev["kind"] >= 3, rng.integers(1, 300, ev.size), 0)
    ev["data_len"][2] = 1500                                     # a burst longer than the stored 1024 bytes
    stored = np.where(ev["kind"] == 3, np.minimum(ev["data_len"], 1024), ev["data_len"])
    perm = rng.permutation(ev.size)                              # payload arena in another order than the events
    start = np.zeros(ev.size, np.int64)
    start[perm] = np.cumsum(stored[perm]) - stored[perm]
    ev["data_offset"] = start
    pay = rng.integers(0, 256, int(stored.sum())).astype(np.uint8)
    limit = 100_000
    k, nev = bench.dump_outputs(str(tmp_path / "a"), ev, pay, ns, max_bytes=limit)
    bench.dump_outputs(str(tmp_path / "b"), ev, pay, ns, max_bytes=limit)
    d, d2 = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert all(np.array_equal(d[x], d2[x]) for x in d)
    assert 0 < k < ns and nev == k * per
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    s = d["streams"].astype(np.int64)
    assert s.size == k and np.all(np.diff(s) > 0) and np.array_equal(np.unique(d["event_stream"]), s)
    for i in range(nev):
        j = int(d["event_stream"][i]) * per + int(d["event_seq"][i])
        o, n = int(d["event_data_offset"][i]), int(stored[j])
        assert d["event_data_len"][i] == ev["data_len"][j]
        assert np.array_equal(d["payload"][o:o + n], pay[ev["data_offset"][j]:ev["data_offset"][j] + n])
    assert d["payload"].size == int(stored[np.isin(ev["stream"], s)].sum())


def test_steps_and_warmup_are_validated():
    for args in (["--steps", "0"], ["--warmup", "-1"]):
        r = _run("--impl", "reference", *args, "--streams", "2", "--seconds", "5")
        assert r.returncode != 0 and "--steps must be" in r.stderr


def test_product_arm_without_gpu_fails_loudly():
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    r = _run("--steps", "1", "--warmup", "3", "--streams", "4", "--seconds", "5", "--no-cpu", "--no-e2e")
    assert r.returncode != 0
    assert r.stdout.strip() == "" or not r.stdout.strip().splitlines()[-1].startswith("{")

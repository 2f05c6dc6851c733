"""The C++ host layer's stream-state calls (include/same_receiver.hpp: export_state / clone / from_state): builds
everywhere; on the GPU a receiver cloned mid-recording and its original both print the golden text."""
import gzip
import os
import subprocess

import pytest

import sameold_b200 as sb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    lib = sb.build_native()
    exe = str(tmp_path / "test_state")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"), "-o", exe,
           os.path.join(ROOT, "tests", "cpp", "test_state.cpp"), "-L" + os.path.dirname(lib), "-lsame_b200",
           "-Wl,-rpath," + os.path.dirname(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    p = tmp_path / "npt.bin"
    with gzip.open(os.path.join(ROOT, "tests", "golden", "npt.22050.s16le.bin.gz"), "rb") as f:
        p.write_bytes(f.read())
    with open(os.path.join(ROOT, "tests", "golden", "npt.22050.s16le.txt")) as f:
        want = [l.rstrip("\n") for l in f if not l.startswith("+OK")]
    assert len(want) == 1
    return exe, str(p), want[0]


def test_cpp_state_layer_builds(tmp_path):
    _build(tmp_path)


@pytest.mark.gpu
def test_cpp_clone_mid_recording_prints_the_golden_text(tmp_path):
    exe, rec, want = _build(tmp_path)
    r = subprocess.run([exe, rec, want], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "CPP_STATE_OK" in r.stdout

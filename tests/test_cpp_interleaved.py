"""The C++ host layer's interleaved entry point (include/same_receiver.hpp, SameBatchReceiver::process_interleaved):
builds everywhere; without a GPU it refuses with SAME_ERR_NO_DEVICE; on the GPU a stereo s16 buffer with the golden
long_message recording in both channels prints samedec's line on both streams."""
import gzip
import os
import subprocess

import pytest

import sameold_b200 as sb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    lib = sb.build_native()
    exe = str(tmp_path / "test_interleaved")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"), "-o", exe,
           os.path.join(ROOT, "tests", "cpp", "test_interleaved.cpp"), "-L" + os.path.dirname(lib), "-lsame_b200",
           "-Wl,-rpath," + os.path.dirname(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    p = tmp_path / "long_message.bin"
    with gzip.open(os.path.join(ROOT, "tests", "golden", "long_message.22050.s16le.bin.gz"), "rb") as f:
        p.write_bytes(f.read())
    return exe, str(p)


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_have_gpu(), reason="checks the no-GPU failure mode")
def test_cpp_interleaved_builds_and_refuses_without_gpu(tmp_path):
    exe, rec = _build(tmp_path)
    r = subprocess.run([exe, rec], capture_output=True, text=True)
    assert r.returncode == 3, (r.returncode, r.stderr)
    assert "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_cpp_interleaved_stereo_long_message(tmp_path):
    exe, rec = _build(tmp_path)
    r = subprocess.run([exe, rec], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "CPP_INTERLEAVED_OK" in r.stdout
    lines = [l for l in r.stdout.splitlines() if l.startswith("stream ")]
    assert len(lines) == 2 and lines[0].split(": ", 1)[1] == lines[1].split(": ", 1)[1]

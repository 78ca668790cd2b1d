"""not-gpu: pins the hand-written DEFLATE encoder (gridfour_b200/csrc/g4_deflate_enc.cuh) byte for byte against the
system zlib by compiling the header's host code path (tests/host/deflate_vs_zlib.cu, nvcc -x cu, -lz).

The reference reaches zlib through java.util.zip (CodecDeflate.java:204-213, CodecFloat.java:268-283,
LsEncoder12.java:180-196); zlib is not part of /root/reference, so the encoder restates zlib's published
deflate_slow / trees.c algorithm and this harness proves the restatement reproduces zlib's bytes for levels 6 and 9
on incompressible, residual-like, run-heavy, multi-block (> 16383 symbols) and multi-window (> 64 KiB) inputs,
including the reference's truncate-at-capacity behaviour."""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
# the nvcc gridfour_b200/csrc/Makefile builds with: PATH first, then the toolkit at CUDA_HOME
NVCC = shutil.which("nvcc") or shutil.which(os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"))


@pytest.mark.skipif(NVCC is None, reason="no nvcc on PATH or under CUDA_HOME")
def test_deflate_encoder_matches_zlib_bytes(tmp_path):
    exe = str(tmp_path / "deflate_vs_zlib")
    subprocess.check_call([NVCC, "-Wno-deprecated-gpu-targets", "-x", "cu", "-O2", "-std=c++17", "-o", exe,
                           os.path.join(HERE, "host", "deflate_vs_zlib.cu"), "-lz"])
    r = subprocess.run([exe, "140000"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
    assert " 0 mismatches" in r.stdout, r.stdout[-2000:]

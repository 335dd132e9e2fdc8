"""The two-class SWAR words of the scan kernel (skywalking-banyandb_b200/csrc/lane_decode.cuh) and the chunk walk that falls back
to the three-class words: tests/native/swar_two_class_test.cc emulates swar_chunk and the masked pass of delta_page_sum_masked
on the host over pages with 3- and 4-byte varints at page, lane and chunk edges, and checks sums, terminator counts, the `wide`
bail-out and which chunks are decoded twice.  No GPU."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_class_chunk_walk_equals_the_three_class_decoder(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    cuda_inc = next((p for p in ("/usr/local/cuda/include", "/usr/local/cuda/targets/x86_64-linux/include") if os.path.exists(os.path.join(p, "vector_types.h"))), None)
    if cuda_inc is None:
        pytest.skip("no CUDA headers (vector_types.h)")
    exe = tmp_path / "swar_two_class_test"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "skywalking-banyandb_b200", "csrc"), "-I", cuda_inc, "-o", str(exe),
                           os.path.join(ROOT, "tests", "native", "swar_two_class_test.cc")])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.startswith("OK"), out.stdout[-2000:] + out.stderr[-2000:]

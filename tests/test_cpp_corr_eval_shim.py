"""The C++ shim of CorrEval (include/vwb200/CorrEval.h): compiles as C++14 against the VW stand-ins and, on a GPU,
reproduces the oracle bit for bit, tile by tile from several threads."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "build", "test_corr_eval_shim")


def _build():
    from visionworkbench_b200 import build
    from oracle import corr_eval
    build.build()
    corr_eval.build()
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    src = os.path.join(ROOT, "tests", "cpp", "test_corr_eval_shim.cpp")
    deps = [src] + [os.path.join(ROOT, "include", "vwb200", f) for f in ("PyramidCorrelationView.h", "CorrEval.h", "vw_standin.h")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-std=c++14", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                               "-L", os.path.join(ROOT, "visionworkbench_b200"), "-lvwb200",
                               os.path.join(ROOT, "oracle", "libvwcorreval.so"), "-lpthread",
                               "-Wl,-rpath," + os.path.join(ROOT, "visionworkbench_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle")])
    return EXE


def test_corr_eval_shim_compiles_as_cxx14_and_fails_loudly_without_a_device():
    exe = _build()
    import visionworkbench_b200 as v
    if v.device_count() > 0:
        pytest.skip("device present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3, r.stdout + r.stderr
    assert "no CUDA device" in r.stdout


@pytest.mark.gpu
def test_corr_eval_shim_matches_oracle_from_threads():
    exe = _build()
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "corr_eval shim: 0 mismatches" in r.stdout, r.stdout

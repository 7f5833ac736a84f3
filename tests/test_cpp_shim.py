"""The C++ drop-in shim (include/vwb200/PyramidCorrelationView.h): compiles against the VW stand-ins,
keeps the lazy-view API, and (on the GPU box) reproduces the oracle tile by tile from several threads."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "build", "test_shim")


def _build():
    from visionworkbench_b200 import build
    import oracle
    build.build()
    oracle.build()
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    src = os.path.join(ROOT, "tests", "cpp", "test_shim.cpp")
    deps = [src] + [os.path.join(ROOT, "include", "vwb200", f) for f in ("PyramidCorrelationView.h", "ParabolaSubpixelView.h", "vw_standin.h")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-std=c++14", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                               "-L", os.path.join(ROOT, "visionworkbench_b200"), "-lvwb200",
                               "-L", os.path.join(ROOT, "oracle"), "-lvworacle", "-lpthread",
                               "-Wl,-rpath," + os.path.join(ROOT, "visionworkbench_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle")])
    return EXE


def test_shim_signature_matches_the_reference_header():
    """The shim's constructor and factory take exactly the parameters of PyramidCorrelationView / pyramid_correlate
    (Stereo/CorrelationView.h:48-69, :195-218): same names, order, defaults, and types from the 5th parameter on (the first
    four are the image views, which the shim takes as ImageViewBase<> templates).  The parameter lists of the reference
    header are stored in tests/golden/pyramid_correlate_signature.json (tests/golden/make_signature.py)."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("make_signature", os.path.join(ROOT, "tests", "golden", "make_signature.py"))
    ms = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ms)
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "pyramid_correlate_signature.json")))
    shim = open(os.path.join(ROOT, "include", "vwb200", "PyramidCorrelationView.h")).read()
    shim = shim[shim.index("class B200PyramidCorrelationView"):]
    ours = {"constructor": ms.param_list(shim, "  B200PyramidCorrelationView("), "factory": ms.param_list(shim, "b200_pyramid_correlate(")}
    for which in ("constructor", "factory"):
        a, b = ours[which], golden[which]
        assert len(a) == len(b) == 24, (which, len(a), len(b))
        assert [q["name"] for q in a] == [q["name"] for q in b], which
        assert [q["default"] for q in a] == [q["default"] for q in b], which
        assert [q["type"] for q in a[4:]] == [q["type"] for q in b[4:]], which


def test_shim_compiles_as_cxx14_and_fails_loudly_without_a_device():
    exe = _build()                     # -std=c++14 like the reference (CMakeLists.txt:20)
    import visionworkbench_b200 as v
    if v.device_count() > 0:
        pytest.skip("device present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3, r.stdout + r.stderr
    assert "no CUDA device" in r.stdout


@pytest.mark.gpu
def test_shim_matches_oracle_from_threads():
    exe = _build()
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "shim: 0 mismatches" in r.stdout and "subpixel shim: 0 mismatches" in r.stdout, r.stdout

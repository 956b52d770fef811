"""mlb::VoiceRouter (include/mlb200_events.hpp) + Voice bank == the complete reference EventsToSignals
on MIDI and MPE phrases (tests/cpp/test_router.cpp).  CPU: bank = the C port.  GPU: bank = the CUDA kernel.

The reference's rows are hashed per phrase in tests/golden/router_digests.txt.  With MLB_RECORD_REFERENCE set
where oracle/_ref/libmle2s.so is built, the test runs the reference beside ours and records the hashes again."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "test_router")
DIGESTS = os.path.join(ROOT, "tests", "golden", "router_digests.txt")


def recording():
    from oracle import bindings
    return bool(os.environ.get("MLB_RECORD_REFERENCE")) and os.path.exists(bindings.E2S_LIB)


def build_exe():
    from madronalib_b200 import api, build
    from oracle import bindings
    if not os.path.exists(api.LIB_PATH):
        build.build()
    if not os.path.exists(bindings.PORT_LIB):
        bindings.build("port")
    dirs = [os.path.dirname(bindings.PORT_LIB), os.path.dirname(api.LIB_PATH)]
    cmd = ["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_router.cpp"), "-o", EXE, "-lmlport", "-lmlb200"]
    if recording():
        dirs.append(os.path.dirname(bindings.E2S_LIB))
        cmd += ["-DHAVE_REFERENCE", "-lmle2s"]
    for d in dirs:
        cmd += ["-L", d, "-Wl,-rpath," + d]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def test_router_plus_port_bank_equals_reference_events_to_signals():
    build_exe()
    r = subprocess.run([EXE, DIGESTS] + (["record"] if recording() else []), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL PASSED" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_router_plus_gpu_bank_equals_reference_events_to_signals(gpu):
    build_exe()
    r = subprocess.run([EXE, DIGESTS, "gpu"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL PASSED" in r.stdout, r.stdout + r.stderr

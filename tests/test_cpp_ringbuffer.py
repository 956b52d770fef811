"""Host-side ring buffer + batched SignalProcessBuffer shim (SURVEY 8f-1): CPU-only C++ test against the
reference's own DSPBuffer: per-run hashes of everything it read back, recorded in
tests/golden/ringbuffer_digests.txt (tests/cpp/lockstep_digest.h).  Where MLB_REFERENCE names the reference
sources, both classes also run in lockstep, and with MLB_RECORD_REFERENCE set the hashes are recorded again."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("MLB_REFERENCE", "")
DIGESTS = os.path.join(ROOT, "tests", "golden", "ringbuffer_digests.txt")


def test_ringbuffer_and_batched_process_buffer():
    exe = os.path.join(ROOT, "tests", "cpp", "test_ringbuffer")
    cmd = ["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_ringbuffer.cpp"), "-o", exe]
    have_ref = bool(REF) and os.path.isdir(os.path.join(REF, "source", "DSP"))
    if have_ref:
        cmd += ["-DHAVE_REFERENCE", "-fno-strict-aliasing", "-include", "cstdint", "-include", "cstddef",
                "-I", os.path.join(REF, "source", "DSP"), "-I", os.path.join(REF, "source", "app"),
                "-I", os.path.join(REF, "include"), "-I", os.path.join(REF, "external")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    record = ["record"] if have_ref and os.environ.get("MLB_RECORD_REFERENCE") else []
    r = subprocess.run([exe, DIGESTS] + record, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ALL PASSED" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    assert "checked in lockstep with the reference" in r.stdout if have_ref else \
        "checked against the reference's recorded digests" in r.stdout

"""mlb::PublishedSignal (include/mlb200_host.hpp) against the reference's own class (CPU-only).

The test compares with per-run hashes of everything the reference's PublishedSignal read back, recorded in
tests/golden/published_digests.txt (tests/cpp/lockstep_digest.h).  Where MLB_REFERENCE names the reference
sources, both classes also run in lockstep, and with MLB_RECORD_REFERENCE set the hashes are recorded again."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("MLB_REFERENCE", "")
DIGESTS = os.path.join(ROOT, "tests", "golden", "published_digests.txt")


def test_published_signal_lockstep_with_reference(tmp_path):
    have_ref = bool(REF) and os.path.isdir(os.path.join(REF, "source", "app"))
    exe = str(tmp_path / "test_published")
    cmd = ["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_published.cpp"), "-o", exe, "-lpthread"]
    if have_ref:
        cmd += ["-DHAVE_REFERENCE", "-fno-strict-aliasing", "-include", "cstdint", "-include", "cstddef",
                "-include", "mutex", "-include", "cstring"]
        for d in ("include", "source/DSP", "source/app", "source/matrix", "external", "external/utf", "external/ffft",
                  "external/aes256", "external/cJSON", "external/sse2neon"):
            cmd += ["-I", os.path.join(REF, d)]
        cmd += [os.path.join(REF, "source/app/MLSignalProcessor.cpp"), os.path.join(REF, "source/app/MLText.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    record = ["record"] if have_ref and os.environ.get("MLB_RECORD_REFERENCE") else []
    r = subprocess.run([exe, DIGESTS] + record, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ALL PASSED" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]

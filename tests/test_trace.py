"""The tracing layer (include/mlb200_trace.hpp): the reference's own example process functions
(examples/audio-and-midi/sine.cpp, reverb.cpp), compiled with only the namespace changed
(tests/cpp/test_trace.cpp), must record graphs that ARE those examples.

CPU part: the traced graph is rebuilt here from its JSON dump and evaluated by the CPU checkers;
the reverb must equal the example's own per-vector body run on the compiled reference
(mlref_aaltoverb).  GPU part: the same binaries run the graphs on the device.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from madronalib_b200.graph import GraphSpec
from tests.common import assert_same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "test_trace")


def build_exe():
    from madronalib_b200 import api, build
    if not os.path.exists(api.LIB_PATH):
        build.build()
    libdir = os.path.dirname(api.LIB_PATH)
    src = os.path.join(ROOT, "tests", "cpp", "test_trace.cpp")
    gen = os.path.join(ROOT, "tests", "cpp", "make_example_bodies.py")
    if os.path.isdir("/root/reference/examples") and not os.path.exists(
            os.path.join(ROOT, "tests", "cpp", "_ref", "reverb_body.inc")):
        subprocess.run([sys.executable, gen], check=True)  # the reference's example bodies: generated, never committed
    hdrs = [os.path.join(ROOT, "include", h) for h in ("mlb200_trace.hpp", "mlb200.hpp", "mlb200_host.hpp", "mlb200.h")]
    hdrs += [os.path.join(ROOT, "tests", "cpp", f) for f in ("kitchen_body.h", "upsample_body.h", "fdn_body.h", "rows_body.h", "rest_body.h", "oversample_body.h")]
    hdrs += [p for p in (os.path.join(ROOT, "tests", "cpp", "_ref", f) for f in ("sine_body.inc", "reverb_body.inc"))
             if os.path.exists(p)]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) > os.path.getmtime(p) for p in [src] + hdrs):
        return
    cmd = ["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
           "-L", libdir, "-lmlb200", "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def traced(case: str, n_voices: int = 1):
    """-> (GraphSpec, coef [n_coef][V], state [n_state][V]) of the graph test_trace records for `case`."""
    build_exe()
    r = subprocess.run([EXE, "dump", case], capture_output=True, text=True, timeout=60)
    if r.returncode == 4:
        pytest.skip("the reference's example bodies were not generated (tests/cpp/make_example_bodies.py needs /root/reference)")
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.loads(r.stdout)
    g = GraphSpec()
    coef_words, state_words = [], []
    for n in d["nodes"]:
        g.ops.append(n["op"])
        g.ins.append(tuple(n["in"]))
        g.iargs.append(n["iarg"])
        coef_words += n["coef"]
        state_words += n["state"]
    g.outs = list(d["outs"])
    coef = np.repeat(np.array(coef_words, np.uint32).view(np.float32)[:, None], n_voices, 1)
    state = np.repeat(np.array(state_words, np.uint32)[:, None], n_voices, 1)
    assert coef.shape[0] == g.n_coef and state.shape[0] == g.n_state and g.n_in == d["n_in"]
    return g, np.ascontiguousarray(coef), np.ascontiguousarray(state)


def test_chain_trace_is_the_survey_plumbing_chain(ref, port):
    """0.5 * Lopass{makeCoeffs(0.1, 1.0)}(SineGen.clear()(440/48000)): SURVEY 8c pinned values."""
    g, coef, state = traced("chain")
    for O in (ref, port):
        out, _, _ = O.run(g, 1, 2, None, state, coef)
        y = out[0, 0, 0]
        assert float(y[0]).hex() == "-0x1.09e6400000000p-9"
        assert float(y[1]).hex() == "-0x1.5cd8fa0000000p-7"
        assert float(y[63]).hex() == "0x1.b253900000000p-3"


def test_sine_example_trace(ref):
    """sine.cpp:29-35: two default-constructed SineGens (phase 0) at 220 and 275 Hz, times 0.1."""
    g, coef, state = traced("sine")
    out, _, _ = ref.run(g, 1, 5, None, state, coef)
    m = GraphSpec()
    for f in (220.0, 275.0):
        m.output(m.node("MULTIPLY", m.node("SINE", m.param()), m.param()))
    mc, ms = m.new_coefs(1), m.new_state(1)
    mc[:, 0] = [np.float32(220.0) / np.float32(48000), np.float32(0.1), np.float32(275.0) / np.float32(48000),
                np.float32(0.1)]
    want, _, _ = ref.run(m, 1, 5, None, ms, mc)
    assert_same_bits(out, want, "sine example")
    assert np.abs(out).max() > 0.09


def reverb_input(T, V=1):
    rng = np.random.default_rng(12)
    x = (rng.standard_normal((T, 2, 1, 64)) * 0.25).astype(np.float32)
    x[6:] = 0  # a burst, then the tail
    return np.ascontiguousarray(np.repeat(x, V, axis=2))


def test_reverb_example_trace_equals_the_example_body(ref, port):
    """reverb.cpp:68-123 traced (two passes find mvFeedbackL/R) == the same body run on the compiled
    reference with its own functor members (mlref_aaltoverb)."""
    g, coef, state = traced("reverb")
    names = [n for n in g.ops]
    assert names.count(108) == 2 and names.count(109) == 2 and names.count(107) == 10  # FEEDBACK_READ/WRITE, ALLPASS_PB
    T = 40
    x = reverb_input(T)
    fb = wl.aaltoverb_feedback(0.5, 0.5)
    want, _ = ref.aaltoverb(x[:, :, 0], 1.0, fb, 0.1 * 48000)
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "traced Aaltoverb vs the example body")
    assert np.abs(want[20:]).max() > 1e-3  # the tail rings


def test_shelf_trace_port_equals_reference(ref, port):
    """vcoeffs -> RAMP x 5 -> LOSHELF_V, Bank<SineGen, 2>, NoiseGen: both checkers agree on the traced graph."""
    g, coef, state = traced("shelf", 3)
    x = np.full((6, 1, 3, 64), 0.013, np.float32)
    ro, _, _ = ref.run(g, 3, 6, x, state, coef)
    po, _, _ = port.run(g, 3, 6, x, state, coef)
    assert_same_bits(po, ro, "shelf trace")
    assert np.isfinite(ro).all() and np.abs(ro).max() > 1e-3


def kitchen_input(T, V=1):
    """gate row (amplitude 0.8 while ((n mod 900) < 500), else 0) and a slowly moving frequency row."""
    n = np.arange(T * 64).reshape(T, 1, 1, 64)
    gate = (((n % 900) < 500) * np.float32(0.8)).astype(np.float32)
    freq = (np.float32(220.0 / 48000.0) * (1.0 + 0.1 * np.sin(n * 0.001))).astype(np.float32)
    x = np.concatenate([gate, freq], axis=1)
    return np.ascontiguousarray(np.repeat(x, V, axis=2))


def test_kitchen_body_same_source_same_bits(ref, port):
    """tests/cpp/kitchen_body.h -- ONE source file, compiled against the reference (`using namespace ml;`, inside
    oracle/ref/mlref.cpp) and against the tracing layer (`using namespace mlb::tr;`): every generator, the SVF family,
    one-poles, ADSR, followers, glides, delays, Allpass<IntegerDelay>, vcoeffs, compound assignment, a carried
    DSPVector member.  The traced graph evaluated by either checker equals the reference build of the same source."""
    g, coef, state = traced("kitchen")
    T = 40
    x = kitchen_input(T)
    want = ref.kitchen(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "kitchen body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want).max() > 0.05


def upsample_input(T, V=1):
    """a slowly moving frequency row (original rate) and a gate row"""
    n = np.arange(T * 64).reshape(T, 1, 1, 64)
    freq = (np.float32(330.0 / 48000.0) * (1.0 + 0.2 * np.sin(n * 0.0007))).astype(np.float32)
    gate = (((n % 700) < 450) * np.float32(0.9)).astype(np.float32)
    x = np.concatenate([freq, gate], axis=1)
    return np.ascontiguousarray(np.repeat(x, V, axis=2))


def test_upsample_body_same_source_same_bits(ref, port):
    """tests/cpp/upsample_body.h -- ONE source, compiled against the reference and against the tracing layer: a process
    function WITH STATE (SineGen, SawGen, Lopass, Bell, OnePole, ADSR, LinearGlide) run twice per vector by
    Upsample2xFunction<1> (the tracing layer records the second run as MLB_AGAIN nodes), and a stateless one run at half
    the rate by Downsample2xFunction<1>; the traced graph evaluated by either checker equals the reference build of the
    same source."""
    from madronalib_b200.graph import OP_NAME
    g, coef, state = traced("upsample")
    again = [i for i in range(g.n_nodes) if g.again_target(i) >= 0]
    assert sorted(OP_NAME[g.ops[i]] for i in again) == ["ADSR", "BELL", "GLIDE", "LOPASS", "ONEPOLE", "SAW", "SINE"]
    assert all(OP_NAME[g.ops[i]] != "NOISE" for i in again)  # called once per vector, outside fn
    assert [OP_NAME[op] for op in g.ops].count("DOWN2X_IN") == 1 and g.n_out == 2
    T = 40
    x = upsample_input(T)
    want = ref.upsample_body(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "upsample body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want).max() > 0.05


def test_fdn_body_same_source_same_bits(ref, port):
    """tests/cpp/fdn_body.h -- ONE source, compiled against the reference and against the tracing layer: FDN<4> and FDN<6>
    (MLDSPFilters.h:1162-1239; the device has one fused node for FDN<8> only).  The tracing layer records them as the
    IntegerDelays, OnePoles, sums and feedback edges they are made of; the traced graph evaluated by either checker
    equals the reference build of the same source."""
    from madronalib_b200.graph import OP_NAME
    g, coef, state = traced("fdn")
    names = [OP_NAME[op] for op in g.ops]
    assert names.count("INTEGER_DELAY") == 10 and names.count("ONEPOLE") == 10
    assert names.count("FEEDBACK_READ") == 10 and names.count("FEEDBACK_WRITE") == 10 and "FDN8" not in names
    T = 60
    x = reverb_input(T)
    want = ref.fdn_body(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "fdn body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want).max() > 0.05 and np.sqrt((want[-10:] ** 2).mean()) > 1e-8  # a decaying tail


def test_rows_body_same_source_same_bits(ref, port):
    """tests/cpp/rows_body.h -- ONE source, compiled against the reference and against the tracing layer:
    DSPVectorArray<ROWS> as a value (rowwise + - * / and compound forms), every row operation of MLDSPOps.h:1056-1383,
    rowIndex / columnIndex / rangeOpen / rangeClosed, Bank<T, ROWS> with array arguments, the "1" forms, the array lerp,
    comparisons, select, int <-> float conversions, int arithmetic (a symbolic DSPVectorInt)."""
    g, coef, state = traced("rows")
    T = 30
    n = np.arange(T * 64).reshape(T, 1, 1, 64)
    x = (np.float32(110.0 / 48000.0) * (1.0 + 0.3 * np.sin(n * 0.002))).astype(np.float32)
    want = ref.rows_body(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "rows body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want[:, 0]).max() > 0.1 and np.abs(want[:, 1]).max() > 0.05


def rest_input(T, V=1):
    """a noise burst (then silence) and a delay-time row sweeping 70 .. 330 samples"""
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((T, 1, 1, 64)) * 0.3).astype(np.float32)
    x[T // 2:] = 0
    n = np.arange(T * 64).reshape(T, 1, 1, 64)
    d = (np.float32(200.0) + np.float32(130.0) * np.sin(n * 0.0031)).astype(np.float32)
    return np.ascontiguousarray(np.repeat(np.concatenate([x, d], axis=1), V, axis=2))


def test_rest_body_same_source_same_bits(ref, port):
    """tests/cpp/rest_body.h -- ONE source, compiled against the reference and against the tracing layer: ImpulseGen,
    OneShotGen, Interpolator1, Allpass1, Differentiator, FractionalDelay (fixed and per-sample), IntegerDelay
    (per-sample), Allpass<FractionalDelay>, PitchbendableDelay used directly, and the fused FDN<8> node."""
    from madronalib_b200.graph import OP_NAME
    g, coef, state = traced("rest")
    names = {OP_NAME[op] for op in g.ops}
    assert {"IMPULSE", "ONESHOT", "INTERPOLATOR1", "ALLPASS1", "DIFFERENTIATOR", "FRACTIONAL_DELAY", "FRACTIONAL_DELAY_VAR",
            "INTEGER_DELAY_VAR", "ALLPASS_FRAC", "PITCHBEND_DELAY", "FDN8", "FDN8_R"} <= names
    T = 48
    x = rest_input(T)
    want = ref.rest_body(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "rest body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want).max() > 0.05 and np.abs(want[-6:]).max() > 1e-6


def test_oversample_body_same_source_same_bits(ref, port):
    """tests/cpp/oversample_body.h -- ONE source, compiled against the reference and against the tracing layer: oversampled
    loops inside one process call between an Upsampler and a Downsampler (MLDSPFilters.h:1316-1473), 4x and 2x, with
    functors that run at the high rate (called four / two times per vector) and an oscillator called twice in a vector.
    Every repeated call is an MLB_AGAIN node, the half-band filters of the cascades included."""
    from madronalib_b200.graph import OP_NAME
    g, coef, state = traced("oversample")
    again = sorted(OP_NAME[g.ops[i]] for i in range(g.n_nodes) if g.again_target(i) >= 0)
    assert again == sorted(["LOPASS"] * 3 + ["ONEPOLE"] * 3 + ["DCBLOCKER"] + ["SINE"] + ["HALFBAND_UP"] + ["HALFBAND_DOWN"])
    T = 36
    rng = np.random.default_rng(9)
    x = (rng.standard_normal((T, 1, 1, 64)) * 0.4).astype(np.float32)
    want = ref.oversample_body(x[:, :, 0])
    for O in (ref, port):
        out, _, _ = O.run(g, 1, T, x, state, coef)
        assert_same_bits(out[:, :, 0], want, "oversample body: traced graph vs the reference build of the same source")
    assert np.isfinite(want).all() and np.abs(want[:, 0]).max() > 0.1 and np.abs(want[:, 1]).max() > 0.05


def test_what_cannot_be_called_twice_is_refused():
    """a functor with a delay ring called twice in a vector (its ring is written once per vector), and a functor inside
    the process function of a Downsample2xFunction"""
    build_exe()
    r = subprocess.run([EXE, "dump", "twice"], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "cannot be called again" in (r.stdout + r.stderr)
    r = subprocess.run([EXE, "dump", "halfrate"], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "must be stateless" in (r.stdout + r.stderr)


def _run_gpu_case(tmp_path, case, V, T, inp):
    build_exe()
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    if inp is not None:
        inp.tofile(fin)
    r = subprocess.run([EXE, "run", case, str(V), str(T), fin, fout], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("case,V,T", [("chain", 70, 6), ("sine", 33, 4), ("reverb", 37, 24), ("shelf", 40, 5),
                                      ("kitchen", 35, 20)])
def test_traced_examples_on_gpu(gpu, port, ref, tmp_path, case, V, T):
    O = ref
    g, coef, state = traced(case, V)
    inp = None
    if case == "reverb":
        inp = reverb_input(T, V)
    if case == "shelf":
        inp = np.ascontiguousarray(np.broadcast_to((0.001 * (1 + np.arange(V, dtype=np.float32)))[None, None, :, None],
                                                   (T, 1, V, 64)))
    if case == "kitchen":
        inp = kitchen_input(T, V)
    _run_gpu_case(tmp_path, case, V, T, inp)
    got = np.fromfile(str(tmp_path / "out.bin"), np.float32).reshape(T, g.n_out, V, 64)
    want, _, _ = O.run(g, V, T, inp, state, coef)
    if case == "kitchen":
        # output 1 is built on Peak / RMS (the CPU's 12-bit rsqrt approximation): tolerance-only off the CPU
        assert_same_bits(got[:, 0], want[:, 0], "kitchen output 0 traced on the GPU")
        assert np.abs(got[:, 1] - want[:, 1]).max() <= 2e-3 * np.abs(want[:, 1]).max()
        assert_same_bits(got[:, 0, 7], O.kitchen(inp[:, :, 0])[:, 0], "GPU vs the reference build of kitchen_body.h")
        return
    assert_same_bits(got, want, case + " traced on the GPU")
    if case == "reverb":
        body, _ = O.aaltoverb(inp[:, :, 0], 1.0, wl.aaltoverb_feedback(0.5, 0.5), 0.1 * 48000)
        assert_same_bits(got[:, :, 5], body, "GPU vs the reverb example's own body")


@pytest.mark.gpu
def test_signal_process_buffer_shaped_streaming_on_gpu(gpu, port, tmp_path):
    """TracedProcessor::process = SignalProcessBuffer::process (MLSignalProcessBuffer.cpp:36-90): host buffers
    of 37 / 100 / 512 / 64 / 1 / 333 frames, one launch per call; the delivered stream equals the vectors
    computed block by block (the sine example: no inputs, so no input-ring latency enters)."""
    build_exe()
    frames = 3000
    g, coef, state = traced("sine", 1)
    fout = str(tmp_path / "out.bin")
    r = subprocess.run([EXE, "stream", "sine", str(frames), "-", fout], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(fout, np.float32).reshape(2, frames)
    T = (frames + 63) // 64
    want, _, _ = port.run(g, 1, T, None, state, coef)
    want = want[:, :, 0].transpose(1, 0, 2).reshape(2, T * 64)[:, :frames]
    assert_same_bits(got, want, "streamed sine example")

"""GPU parity of the features added after the round's GPU budget was spent: MLB_AGAIN graphs (a functor called again in
the same vector, mlb200.h: a process function with state inside Upsample2xFunction) FDN<SIZE> for sizes other than
8, written out with the nodes it is made of, and the array-valued spellings of the tracing layer.  Collected last (the file name): these tests were written when the round's GPU budget was
nearly spent and were rehearsed on the CPU checkers first; they met the hardware in the round's last, 7-second call
(13 passed, profiles/gpu_tests_late_r2.txt).  The CPU side of the feature: test_abi.py, test_oracle_port_vs_ref.py, test_oracle_golden.py,
test_trace.py."""
import os

import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from tests.common import assert_same_bits, assert_state_equal, run_gpu

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", wl.AGAIN_CASES)
@pytest.mark.parametrize("n_voices", [40, 97])
def test_again_case_bit_exact(gpu, port, name, n_voices):
    w = wl.functor_case(name, n_voices)
    T = 24
    inp = w.inputs(T)
    po, _, ps = port.run(w.spec, n_voices, T, inp, w.state, w.coef)
    go, _, gs, kname = run_gpu(gpu, w, T, inp, splits=(5, 7, 12))
    assert kname.startswith("generic"), kname
    assert_same_bits(go, po, name)
    assert_state_equal(gs, ps, name)


@pytest.mark.parametrize("name", wl.AGAIN_CASES)
def test_again_case_matches_committed_reference_golden(gpu, name):
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "functors.npz"))
    inp = gold[name + "_in"]
    T, V = inp.shape[0], inp.shape[2]
    w = wl.functor_case(name, V)
    w.coef, w.state = gold[name + "_coef"], gold[name + "_state0"]
    go, _, gs, _ = run_gpu(gpu, w, T, inp)
    assert_same_bits(go, gold[name + "_out"], name)
    assert_state_equal(gs, gold[name + "_state1"], name)


@pytest.mark.parametrize("seed", [217, 226, 238])
def test_random_graphs_with_functors_called_again(gpu, port, monkeypatch, seed):
    """MLB_AGAIN on the device: random DAGs in which generators, filters and glides are called again in the same
    vector (the further call reads and writes the words of the first), default stage count and forced cuts (a functor
    and its further calls stay in one stage).  Seeds screened on the CPU: every node's row is finite, so no NaN sign
    enters (see test_random_graphs_bit_exact); the port is pinned to the compiled reference on the same generator
    (test_oracle_port_vs_ref.py::test_random_graphs_with_functors_called_again)."""
    w = wl.random_graph_workload(seed, 41, 28, hw_approx=False, again_prob=0.5)
    g = w.spec
    assert sum(g.again_target(i) >= 0 for i in range(g.n_nodes)) >= 3
    T = 9
    inp = w.inputs(T)
    po, _, ps = port.run(g, w.n_voices, T, inp, w.state, w.coef)
    assert np.isfinite(po).all()
    for stages in (None, 4, 64):
        if stages:
            monkeypatch.setenv("MLB_STAGES", str(stages))
        go, _, gs, kname = run_gpu(gpu, w, T, inp, splits=(4, 5))
        assert kname.startswith("generic"), kname
        assert_same_bits(go, po, "random graph with AGAIN nodes %d (%s)" % (seed, kname))
        assert_state_equal(gs, ps, "random graph with AGAIN nodes %d (%s)" % (seed, kname))


def test_upsample2x_with_a_stateful_process_function_on_the_device(gpu, ref):
    """The reference's own Upsample2xFunction<1> around its own SineGen and Lopass objects (both called twice per
    vector) against the MLB_AGAIN graph on the device."""
    V, T = 70, 20
    w = wl.functor_case("upsample2x_osc", V)
    inp = w.inputs(T)
    go, _, gs, kname = run_gpu(gpu, w, T, inp, splits=(7, 13))
    assert kname.startswith("generic"), kname
    g = w.spec
    from madronalib_b200.graph import OP_NAME
    sine = next(i for i in range(g.n_nodes) if OP_NAME[g.ops[i]] == "SINE")
    c0 = g.coef_slot(next(i for i in range(g.n_nodes) if OP_NAME[g.ops[i]] == "LOPASS"))
    for v in (0, 31, 32, 69):
        o = ref.upsample2x_osc(inp[:, 0, v, :], int(w.state[g.state_slot(sine), v]), w.coef[c0:c0 + 3, v])
        assert_same_bits(go[:, 0, v, :], o, "Upsample2xFunction with a stateful fn, voice %d" % v)


def test_traced_upsample_body_on_gpu(gpu, port, ref, tmp_path):
    """tests/cpp/upsample_body.h traced and run on the device == the traced graph on the checker == the reference build
    of the same source."""
    from tests.test_trace import _run_gpu_case, traced, upsample_input
    V, T = 36, 18
    O = ref
    g, coef, state = traced("upsample", V)
    inp = upsample_input(T, V)
    _run_gpu_case(tmp_path, "upsample", V, T, inp)
    got = np.fromfile(str(tmp_path / "out.bin"), np.float32).reshape(T, g.n_out, V, 64)
    want, _, _ = O.run(g, V, T, inp, state, coef)
    assert_same_bits(got, want, "upsample body traced on the GPU")
    assert_same_bits(got[:, :, 7], O.upsample_body(inp[:, :, 0]), "GPU vs the reference build of upsample_body.h")


@pytest.mark.parametrize("size", [4, 6, 16])
def test_fdn_of_any_size_on_the_device(gpu, port, ref, size):
    """FDN<SIZE> written out with IntegerDelay / OnePole / feedback-edge nodes (graph.graph_fdn) through the interpreter,
    against the port and against the reference's own FDN<SIZE> object."""
    V, T = 45, 30
    w, times, cutoffs, gains = wl.fdn_case(size, V)
    inp = w.inputs(T)
    po, _, ps = port.run(w.spec, V, T, inp, w.state, w.coef)
    go, _, gs, kname = run_gpu(gpu, w, T, inp, splits=(11, 19))
    assert kname.startswith("generic"), kname
    assert_same_bits(go, po, "fdn%d (%s)" % (size, kname))
    assert_state_equal(gs, ps, "fdn%d" % size)
    for v in (0, 44):
        assert_same_bits(go[:, :, v, :], ref.fdn(size, inp[:, 0, v, :], times[:, v], cutoffs, gains), "vs FDN<%d> itself" % size)


def test_traced_fdn_body_on_gpu(gpu, port, ref, tmp_path):
    """tests/cpp/fdn_body.h (FDN<4> + FDN<6>) traced and run on the device == the reference build of the same source."""
    from tests.test_trace import _run_gpu_case, reverb_input, traced
    V, T = 34, 40
    O = ref
    g, coef, state = traced("fdn", V)
    inp = reverb_input(T, V)
    _run_gpu_case(tmp_path, "fdn", V, T, inp)
    got = np.fromfile(str(tmp_path / "out.bin"), np.float32).reshape(T, g.n_out, V, 64)
    want, _, _ = O.run(g, V, T, inp, state, coef)
    assert_same_bits(got, want, "fdn body traced on the GPU")
    assert_same_bits(got[:, :, 5], O.fdn_body(inp[:, :, 0]), "GPU vs the reference build of fdn_body.h")


def test_traced_rows_body_on_gpu(gpu, port, ref, tmp_path):
    """tests/cpp/rows_body.h (DSPVectorArray<ROWS> as a value, the row operations, Bank with array arguments) traced and
    run on the device == the reference build of the same source."""
    from tests.test_trace import _run_gpu_case, traced
    V, T = 33, 12
    O = ref
    g, coef, state = traced("rows", V)
    n = np.arange(T * 64).reshape(T, 1, 1, 64)
    inp = np.ascontiguousarray(np.repeat((np.float32(110.0 / 48000.0) * (1.0 + 0.3 * np.sin(n * 0.002))).astype(np.float32),
                                         V, axis=2))
    _run_gpu_case(tmp_path, "rows", V, T, inp)
    got = np.fromfile(str(tmp_path / "out.bin"), np.float32).reshape(T, g.n_out, V, 64)
    want, _, _ = O.run(g, V, T, inp, state, coef)
    assert_same_bits(got, want, "rows body traced on the GPU")
    assert_same_bits(got[:, :, 9], O.rows_body(inp[:, :, 0]), "GPU vs the reference build of rows_body.h")


def test_traced_oversample_body_on_gpu(gpu, port, ref, tmp_path):
    """tests/cpp/oversample_body.h (4x / 2x oversampled loops between an Upsampler and a Downsampler; functors and the
    half-band stages called several times per vector) traced and run on the device == the reference build of the same
    source.  Written after the round's last GPU call (the other tests of this file ran in it): every device path it
    takes is one they take -- an MLB_AGAIN node is an ordinary node with another node's word offsets -- and its plan is
    checked in test_planner.py; the first hardware run of this particular graph is the round-end one."""
    from tests.test_trace import _run_gpu_case, traced
    V, T = 35, 14
    O = ref
    g, coef, state = traced("oversample", V)
    rng = np.random.default_rng(9)
    inp = np.ascontiguousarray(np.repeat((rng.standard_normal((T, 1, 1, 64)) * 0.4).astype(np.float32), V, axis=2))
    _run_gpu_case(tmp_path, "oversample", V, T, inp)
    got = np.fromfile(str(tmp_path / "out.bin"), np.float32).reshape(T, g.n_out, V, 64)
    want, _, _ = O.run(g, V, T, inp, state, coef)
    assert_same_bits(got, want, "oversample body traced on the GPU")
    assert_same_bits(got[:, :, 11], O.oversample_body(inp[:, :, 0]), "GPU vs the reference build of oversample_body.h")

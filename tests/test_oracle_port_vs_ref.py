"""The plain-C port against the compiled reference on fresh random inputs (the reference's results as
recorded in tests/golden/reference.npz, see tests/recorded_reference.py)."""
import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from madronalib_b200.graph import OP_NAME, OP_TABLE, GraphSpec
from tests.common import assert_state_equal


def test_this_is_the_reference(ref):
    # SURVEY appendix A sizes: DSPVector, Lopass, OnePole, SineGen, IntegerDelay, FDN<8>
    assert [ref.sizeof(i) for i in range(6)] == [256, 20, 12, 4, 48, 2560]


@pytest.mark.parametrize("seed", [0, 1])
def test_all_stateless_ops(ref, port, seed):
    rng = np.random.default_rng(seed)
    V, T = 5, 2
    for name, (_, nin, nst, nco) in OP_TABLE.items():
        if not (30 <= OP_TABLE[name][0] < 100):  # MLB_OP_MAP_FIRST .. MLB_OP_MAP_END
            continue
        g = GraphSpec()
        g.output(g.node(name, *[g.input(k) for k in range(nin)]))
        x = (rng.standard_normal((T, nin, V, 64)) * 10.0 ** rng.integers(-3, 4)).astype(np.float32)
        a, _, _ = ref.run(g, V, T, x, g.new_state(V), g.new_coefs(V))
        b, _, _ = port.run(g, V, T, x, g.new_state(V), g.new_coefs(V))
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name


@pytest.mark.parametrize("make,T", [
    (lambda: wl.config_a(70), 5), (lambda: wl.config_2("bell", 40), 4),
    (lambda: wl.config_2("hishelf", 40), 4), (lambda: wl.config_3(50), 4),
    (lambda: wl.config_4(24), 20), (lambda: wl.config_5(6, 256), 3)])
def test_configs_random_state(ref, port, make, T):
    w = make()
    rng = np.random.default_rng(3)
    st = w.state.copy()
    # start mid-stream: random filter state (phases stay as set)
    for i, op in enumerate(w.spec.ops):
        from madronalib_b200.graph import OP_INFO, OP_NAME
        if OP_NAME[op] in ("LOPASS", "HIPASS", "BANDPASS", "LOSHELF", "HISHELF", "BELL", "ONEPOLE"):
            s0 = w.spec.state_slot(i)
            n = OP_INFO[op][1]
            st[s0:s0 + n] = (rng.standard_normal((n, w.n_voices)) * 0.1).astype(np.float32).view(np.uint32)
    inp = w.inputs(T)
    a, am, ast = ref.run(w.spec, w.n_voices, T, inp, st, w.coef, want_mix=True)
    b, bm, bst = port.run(w.spec, w.n_voices, T, inp, st, w.coef, want_mix=True, nthreads=3)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.array_equal(am.view(np.uint32), bm.view(np.uint32))
    assert_state_equal(ast, bst)


def test_reference_chain_loop_equals_graph(ref):
    """The CPU-baseline loop (struct Voice{SineGen; Lopass}) computes exactly the graph result."""
    w = wl.config_a(64)
    T = 4
    inp = w.inputs(T)
    want, _, _ = ref.run(w.spec, 64, T, inp, w.state, w.coef)
    phase = w.state[0].copy()
    ic = w.state[1:3].view(np.float32).copy()
    got, sec = ref.chain_sine_lopass_gain(np.ascontiguousarray(inp[:, 0]), np.ascontiguousarray(w.coef[0:3]),
                                          np.ascontiguousarray(w.coef[3]), phase, ic, 2)
    assert np.array_equal(got.view(np.uint32), want[:, 0].view(np.uint32)) and sec > 0


@pytest.mark.parametrize("name", wl.FUNCTOR_CASES + wl.AGAIN_CASES)
def test_functor_cases(ref, port, name):
    """SURVEY 8(f) row 2: every added functor, port == compiled reference, bit for bit, with the
    port run split over three calls (state and delay memory carried inside the oracle)."""
    w = wl.functor_case(name, 40)
    T = 24
    inp = w.inputs(T)
    a, _, ast = ref.run(w.spec, w.n_voices, T, inp, w.state, w.coef)
    b, _, bst = port.run(w.spec, w.n_voices, T, inp, w.state, w.coef, splits=(5, 7, 12), nthreads=2)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert_state_equal(ast, bst)
    assert np.abs(a).max() > 0


def test_aaltoverb_graph_is_the_example(ref, port):
    """graph_aaltoverb() == the body of examples/audio-and-midi/reverb.cpp driven directly
    (mlref_aaltoverb), and the port agrees with both."""
    w = wl.config_6(6)
    T = 120
    inp = w.inputs(T)
    a, _, ast = ref.run(w.spec, w.n_voices, T, inp, w.state, w.coef)
    b, _, bst = port.run(w.spec, w.n_voices, T, inp, w.state, w.coef, splits=(50, 70))
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert_state_equal(ast, bst)
    for v in (0, 3, 5):
        size2 = float(w.coef[w.spec.coef_slot(2), v])
        fb = float(w.coef[w.spec.coef_slot(3), v])
        o, _ = ref.aaltoverb(inp[:, :, v, :], size2, fb, 4800.0)
        assert np.array_equal(o.view(np.uint32), a[:, :, v, :].view(np.uint32))
    assert np.sqrt((a[-10:] ** 2).mean()) > 1e-3  # the tail is ringing, not silent


def test_upsample2x_graph_is_the_higher_order_function(ref):
    """HALFBAND_DOWN(fn(HALFBAND_UP(x)), fn(HALFBAND_UP_2(x))) == the reference's Upsample2xFunction<1>
    (MLDSPFunctional.h:114-160) called directly with fn(v) = clamp(v * drive, -1, 1)."""
    w = wl.functor_case("upsample2x_clip", 12)
    T = 20
    inp = w.inputs(T)
    a, _, _ = ref.run(w.spec, 12, T, inp, w.state, w.coef)
    for v in (0, 7, 11):
        o = ref.upsample2x_clip(inp[:, 0, v, :], float(w.coef[0, v]))
        assert np.array_equal(o.view(np.uint32), a[:, 0, v, :].view(np.uint32))


def test_upsample2x_with_a_stateful_process_function(ref, port):
    """MLB_AGAIN: fn(v) = lp(osc(v * 0.5)) run twice per vector by Upsample2xFunction<1> -- the graph in which the
    SINE and LOPASS nodes are called again == the reference's wrapper around its own SineGen and Lopass objects
    (MLDSPFunctional.h:114-160; the tutorial wraps a sine generator this way, dspOpsExample.cpp:100-102)."""
    V, T = 12, 24
    w = wl.functor_case("upsample2x_osc", V)
    g = w.spec
    assert g.n_state == 9 + 1 + 2 + 9 and g.n_coef == 1 + 3   # the AGAIN nodes own no words
    inp = w.inputs(T)
    a, _, sa = ref.run(g, V, T, inp, w.state, w.coef, splits=(5, 19))
    b, _, sb = port.run(g, V, T, inp, w.state, w.coef)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(sa, sb)
    sine = [i for i, op in enumerate(g.ops) if OP_NAME[op] == "SINE"]
    lp = [i for i, op in enumerate(g.ops) if OP_NAME[op] == "LOPASS"]
    assert g.again_target(sine[1]) == sine[0] and g.again_target(lp[1]) == lp[0]
    assert g.state_slot(sine[1]) == g.state_slot(sine[0]) and g.coef_slot(lp[1]) == g.coef_slot(lp[0])
    c0 = g.coef_slot(lp[0])
    for v in (0, 5, 11):
        o = ref.upsample2x_osc(inp[:, 0, v, :], int(w.state[g.state_slot(sine[0]), v]), w.coef[c0:c0 + 3, v])
        assert np.array_equal(o.view(np.uint32), a[:, 0, v, :].view(np.uint32))
    assert np.abs(a).max() > 0.3
    # ticking twice matters: with two independent functors per kind instead, the signal is another one
    h = GraphSpec()
    h.ops, h.ins, h.outs = list(g.ops), list(g.ins), list(g.outs)
    h.iargs = [0 if g.again_target(i) >= 0 else g.iargs[i] for i in range(g.n_nodes)]
    assert h.n_state == g.n_state + 3 and h.n_coef == g.n_coef + 3
    hc, hs = h.new_coefs(V), h.new_state(V)
    hc[h.coef_slot(3)] = 0.5  # the param node
    for n in lp:
        hc[h.coef_slot(n):h.coef_slot(n) + 3] = w.coef[c0:c0 + 3]
    for n in sine:
        hs[h.state_slot(n)] = w.state[g.state_slot(sine[0])]
    c, _, _ = port.run(h, V, T, inp, hs, hc)
    assert not np.array_equal(c, b)


@pytest.mark.parametrize("seed", range(8))
def test_random_graphs_with_functors_called_again(ref, port, seed):
    """Random DAGs in which generators, filters and glides are called AGAIN in the same vector (MLB_AGAIN): the port
    (words shared through the layout) against the compiled reference (the same functor object simply called twice)."""
    w = wl.random_graph_workload(100 + seed, n_voices=9, n_nodes=30, again_prob=0.5)
    g = w.spec
    n_again = sum(g.again_target(i) >= 0 for i in range(g.n_nodes))
    assert n_again >= 2
    T = 12
    inp = w.inputs(T)
    a, _, sa = ref.run(g, 9, T, inp, w.state, w.coef, splits=(5, 7))
    b, _, sb = port.run(g, 9, T, inp, w.state, w.coef)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), seed
    assert_state_equal(sb, sa, "state after, seed %d" % seed)


@pytest.mark.parametrize("size", [4, 6, 8, 16])
def test_fdn_of_any_size_written_out_with_its_parts(ref, port, size):
    """FDN<SIZE> (MLDSPFilters.h:1162-1239) for SIZE other than the fused 8: the graph made of SIZE IntegerDelays, the
    sums, the Householder step, SIZE OnePoles, gains and one-block feedback edges (graph.graph_fdn) == the reference's
    own FDN<SIZE> object, bit for bit, on both checkers (SIZE = 8 included as a cross-check of the recipe)."""
    V, T = 7, 40
    w, times, cutoffs, gains = wl.fdn_case(size, V)
    inp = w.inputs(T)
    a, _, sa = ref.run(w.spec, V, T, inp, w.state, w.coef, splits=(9, 31))
    b, _, sb = port.run(w.spec, V, T, inp, w.state, w.coef)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert_state_equal(sb, sa, "fdn%d" % size)
    for v in (0, 3, 6):
        o = ref.fdn(size, inp[:, 0, v, :], times[:, v], cutoffs, gains)
        assert np.array_equal(o.view(np.uint32), a[:, :, v, :].view(np.uint32)), (size, v)
    assert np.sqrt((a[-8:] ** 2).mean()) > 1e-4  # the tail rings


def test_downsample2x_graph_is_the_higher_order_function(ref):
    """DOWN2X_OUT(fn(DOWN2X_IN(x))) == the reference's Downsample2xFunction<1> (MLDSPFunctional.h:166-223)
    called directly with fn(v) = clamp(v * drive, -1, 1)."""
    w = wl.functor_case("downsample2x_clip", 12)
    T = 21
    inp = w.inputs(T)
    a, _, _ = ref.run(w.spec, 12, T, inp, w.state, w.coef)
    for v in (0, 7, 11):
        o = ref.downsample2x_clip(inp[:, 0, v, :], float(w.coef[0, v]))
        assert np.array_equal(o.view(np.uint32), a[:, 0, v, :].view(np.uint32))


@pytest.mark.parametrize("seed", range(16))
def test_random_graphs(ref, port, seed):
    """Random DAGs over most of the op table (generators, filters, delay functors, feedback edges, elementwise
    ops): the C port and the compiled reference agree bit for bit, NaNs included, with the port run split."""
    w = wl.random_graph_workload(seed, 21, 26)
    T = 9
    inp = w.inputs(T)
    a, _, ast = ref.run(w.spec, w.n_voices, T, inp, w.state, w.coef)
    b, _, bst = port.run(w.spec, w.n_voices, T, inp, w.state, w.coef, splits=(4, 5))
    from tests.common import assert_same_bits
    assert_same_bits(b, a, "random graph %d" % seed)
    assert_state_equal(bst, ast, "random graph %d" % seed)

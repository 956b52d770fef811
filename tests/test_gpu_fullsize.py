"""GPU parity at the BASELINE.json sizes (SURVEY.md 8d), through the DEFAULT launch shapes.

The small-size tests in test_gpu_chain.py cover the edge cases; these cover the shapes bench.py and
tools/bench_configs.py actually time: the persistent 12-warp x 148-CTA chain grid with (group, chunk)
work units and state hopping between warps (only taken above 4 * SMs voice groups), the 16-slice
three-stream host pipeline behind the e2e number, the FDN kernel at 16 384 voices and the graph
interpreter's stage pipeline at 1 024 x 256 nodes.  The checker is the reference itself for rows and state
(as recorded in tests/golden/reference.npz: the port's rows must have the reference's digest), and the port
for the mix bus in the device summation order.
"""
import os

import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from tests.common import assert_same_bits, assert_state_equal

pytestmark = pytest.mark.gpu

NTHREADS = max(1, len(os.sched_getaffinity(0)))


def _device_run(gpu, w, T, inp, want_mix=False, flags=0):
    """One process_device call with HBM-resident buffers (the path bench.py's `value` times)."""
    import torch
    dev = torch.device("cuda", 0)
    g = gpu.VoiceGraph(w.spec, w.n_voices, flags)
    try:
        g.set_coefs(w.coef)
        g.set_state(w.state)
        d_in = torch.from_numpy(inp).to(dev) if inp is not None else None
        d_out = torch.empty((T, w.spec.n_out, w.n_voices, 64), dtype=torch.float32, device=dev)
        d_mix = torch.zeros((T, w.spec.n_out, 64), dtype=torch.float32, device=dev) if want_mix else None
        torch.cuda.synchronize()
        g.process_device(d_in, d_out, d_mix, T, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        out = d_out.cpu().numpy()
        mix = d_mix.cpu().numpy() if want_mix else None
        st = g.get_state()
        name = g.kernel_name
    finally:
        g.close()
    return out, mix, st, name


def test_config_a_full_size_device_path(gpu, port, ref):
    """Config A, 65 536 voices x 64 blocks, default launch shape (W=12 x 148 CTAs, 6 time chunks)."""
    V, T = 65536, 64
    w = wl.config_a(V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    _, pm, _ = port.run(w.spec, V, T, inp, w.state, w.coef, want_out=False, want_mix=True, mix_mode=1,
                        nthreads=NTHREADS)
    go, gm, gs, name = _device_run(gpu, w, T, inp, want_mix=True)
    assert name.startswith("fused:"), name
    assert_same_bits(go, ro, "config A 65536x64 out")
    assert_state_equal(gs, rs, "config A 65536x64 state")
    assert_same_bits(gm, pm, "config A 65536x64 mix (device order)")
    # and within (V-1) eps sum|x| of the reference's strict left-to-right addRows (MLDSPOps.h:1354-1357)
    ref_mix = ro.astype(np.float64).sum(axis=2)
    tol = V * np.finfo(np.float32).eps * np.abs(ro).sum(axis=2).max()
    assert np.abs(gm - ref_mix).max() <= tol


def test_config_a_full_size_host_pipeline(gpu, port, ref, monkeypatch):
    """The same bank through mlb_graph_process_host: 16 voice slices, H2D / kernel / D2H on three
    streams -- the path behind bench.py's e2e number.  Two successive calls (progress words carry)."""
    monkeypatch.delenv("MLB_HOST_SLICES", raising=False)
    V, T = 65536, 64
    w = wl.config_a(V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    _, pm, _ = port.run(w.spec, V, T, inp, w.state, w.coef, want_out=False, want_mix=True, mix_mode=1,
                        nthreads=NTHREADS)
    g = gpu.VoiceGraph(w.spec, V)
    try:
        g.set_coefs(w.coef)
        g.set_state(w.state)
        h = T // 2
        o1, m1 = g.process_host(np.ascontiguousarray(inp[:h]), h, want_out=True, want_mix=True)
        assert g.last_host_slices == 16
        o2, m2 = g.process_host(np.ascontiguousarray(inp[h:]), T - h, want_out=True, want_mix=True)
        assert g.last_host_slices == 16
        gs = g.get_state()
    finally:
        g.close()
    assert_same_bits(np.concatenate([o1, o2]), ro, "config A host pipeline out")
    assert_same_bits(np.concatenate([m1, m2]), pm, "config A host pipeline mix")
    assert_state_equal(gs, rs, "config A host pipeline state")


def test_config_3_full_size(gpu, port, ref):
    V, T = 65536, 64
    w = wl.config_3(V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    go, _, gs, name = _device_run(gpu, w, T, inp)
    assert name.startswith("fused:"), name
    assert_same_bits(go, ro, "config 3 65536x64 out")
    assert_state_equal(gs, rs, "config 3 65536x64 state")


@pytest.mark.parametrize("kind", ["lopass", "bell"])
def test_config_2_full_size(gpu, port, ref, kind):
    V, T = 4096, 64
    w = wl.config_2(kind, V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    go, _, gs, name = _device_run(gpu, w, T, inp)
    assert name.startswith("fused:"), name
    assert_same_bits(go, ro, "config 2 out " + kind)
    assert_state_equal(gs, rs, "config 2 state " + kind)


def test_config_4_full_size(gpu, port, ref):
    """16 384 voices x 16 blocks of 3-op FM -> FDN<8>, in two launches (ring write index carries)."""
    V, T = 16384, 16
    w = wl.config_4(V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    _, pm, _ = port.run(w.spec, V, T, inp, w.state, w.coef, want_out=False, want_mix=True, mix_mode=1,
                        nthreads=NTHREADS)
    go, gm, gs, name = _device_run(gpu, w, T, inp, want_mix=True)
    assert name.startswith("fused:fm3_fdn8"), name
    assert_same_bits(go, ro, "config 4 16384x16 out")
    assert_same_bits(gm, pm, "config 4 16384x16 mix")
    assert_state_equal(gs, rs, "config 4 16384x16 state")
    assert np.abs(go).max() > 0.1


def test_config_5_full_size(gpu, port, ref):
    """1 024 instances x 256-node chain x 16 blocks through the interpreter's stage pipeline."""
    V, T = 1024, 16
    w = wl.config_5(V, 256)
    ro, _, rs = ref.run(w.spec, V, T, None, w.state, w.coef, nthreads=NTHREADS)
    go, _, gs, name = _device_run(gpu, w, T, None)
    assert name.startswith("generic"), name
    assert_same_bits(go, ro, "config 5 1024x256x16 out " + name)
    assert_state_equal(gs, rs, "config 5 state")


def test_config_6_full_size(gpu, port, ref):
    """4 096 Aaltoverb reverbs x 16 blocks (SURVEY 8f row 2) at the benchmarked size."""
    V, T = 4096, 16
    w = wl.config_6(V)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=NTHREADS)
    go, _, gs, name = _device_run(gpu, w, T, inp)
    assert_same_bits(go, ro, "config 6 4096x16 out " + name)
    assert_state_equal(gs, rs, "config 6 state")


@pytest.mark.parametrize("n_blocks,row_mask", [(64, 0x03), (16, 0xFF)])
def test_voice_bank_full_size(gpu, n_blocks, row_mask):
    """EventsToSignals::Voice x 65 536 (the K7 benchmark shapes: pitch+gate rows over 64 vectors, all 8
    rows) against the port on a stride of voices (voices are independent; the whole bank is checked at
    small sizes in test_voice_bank.py)."""
    from oracle import bindings
    V, T = 65536, n_blocks
    ev = wl.voice_events(256, T, seed=2, density=0.10, ctl=0.05)
    ev = np.ascontiguousarray(np.tile(ev, (1, V // 256)))
    prm = wl.voice_bank_params(V)
    vb = gpu.VoiceBank(48000.0, *prm)
    try:
        got = vb.process_host(ev, row_mask)
    finally:
        vb.close()
    sel = np.arange(0, V, 61)  # 1075 voices spread over every warp position
    want, _ = bindings.port_voice_bank().run(48000.0, *(p[sel] for p in prm), np.ascontiguousarray(ev[:, sel]),
                                             nthreads=NTHREADS)
    rows = [r for r in range(8) if row_mask & (1 << r)]
    assert_same_bits(got[:, rows][:, :, sel], want[:, rows], "voice bank 65536 x %d (1075-voice sample)" % T)

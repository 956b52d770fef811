"""SURVEY 8(f) row 3: EventsToSignals::Voice x V.  CPU: the C port against the reference's own Voice
(compiled in place, oracle/_ref/libmle2s.so) and against committed goldens.  GPU: the CUDA bank,
through the C ABI, against the port -- bit for bit on all 8 rows."""
import os

import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from tests.common import assert_same_bits
from tests.recorded_reference import assert_events_to_signals

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "voices.npz")
ROWS = ["pitch", "gate", "voice", "z", "x", "y", "mod", "time"]


@pytest.fixture(scope="module")
def port_bank():
    from oracle import bindings
    return bindings.port_voice_bank()


@pytest.fixture(scope="module")
def ref_bank():
    from tests import recorded_reference
    return recorded_reference.voice_bank()


@pytest.mark.parametrize("sr,seed,flags", [(48000.0, 3, 0), (44100.0, 4, 1), (1000.0, 5, 1)])
def test_port_equals_reference_voice(ref_bank, port_bank, sr, seed, flags):
    """sr = 1000 makes the 8-second drift interval 125 vectors long, so the drift redraw and the drift
    glide run inside the test."""
    V, T = 40, 300
    ev = wl.voice_events(V, T, seed=seed)
    prm = wl.voice_bank_params(V)
    a, _ = ref_bank.run(sr, *prm, ev, flags=flags)
    b, _ = port_bank.run(sr, *prm, ev, splits=(7, 93, 200), flags=flags)
    for r, name in enumerate(ROWS):
        assert np.array_equal(a[:, r].view(np.uint32), b[:, r].view(np.uint32)), name
    assert np.abs(a[:, 0]).max() > 1 and a[:, 1].max() > 0.5 and a[:, 7].max() > 0


def test_port_matches_committed_golden(port_bank):
    g = np.load(GOLD)
    ev = g["events"].view(wl.VOICE_EVENTS_DTYPE).reshape(g["shape"][0], g["shape"][1])
    V = ev.shape[1]
    assert np.array_equal(ev.view(np.uint8), wl.voice_events(V, ev.shape[0], seed=11).view(np.uint8))
    b, _ = port_bank.run(float(g["sr"]), *wl.voice_bank_params(V), ev, flags=wl.VOICES_MIDI)
    assert np.array_equal(b.view(np.uint32), g["out"].view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("sr,V,T,seed,flags", [(48000.0, 70, 120, 6, 0), (1000.0, 33, 300, 7, 1),
                                               (44100.0, 300, 40, 8, 1)])
def test_gpu_voice_bank_bit_exact(gpu, port_bank, sr, V, T, seed, flags):
    ev = wl.voice_events(V, T, seed=seed)
    prm = wl.voice_bank_params(V)
    want, _ = port_bank.run(sr, *prm, ev, flags=flags)
    vb = gpu.VoiceBank(sr, *prm, flags=flags)
    try:
        got = np.concatenate([vb.process_host(ev[:T // 3]), vb.process_host(ev[T // 3:])], axis=0)
    finally:
        vb.close()
    for r, name in enumerate(ROWS):
        assert_same_bits(got[:, r], want[:, r], name)


@pytest.mark.gpu
@pytest.mark.parametrize("mask,flags", [(0x7F, 1), (0x7C, 0), (0x49, 1), (0x80, 0)])
def test_gpu_voice_bank_row_masks(gpu, port_bank, mask, flags):
    """The kernel instance without the elapsed-time row (two tiles, 7 warps per CTA) writing the glide-only rows,
    with and without the MIDI pressure glide; rows that are not wanted still advance their glides (second call)."""
    sr, V, T = 48000.0, 270, 60
    ev = wl.voice_events(V, T, seed=31)
    prm = wl.voice_bank_params(V)
    want, _ = port_bank.run(sr, *prm, ev, flags=flags)
    vb = gpu.VoiceBank(sr, *prm, flags=flags)
    try:
        a = vb.process_host(ev[:T // 2], row_mask=mask)
        b = vb.process_host(ev[T // 2:])  # all rows: every glide must be where the reference's is
    finally:
        vb.close()
    for r, name in enumerate(ROWS):
        if mask & (1 << r):
            assert_same_bits(a[:, r], want[:T // 2, r], "masked call, " + name)
        else:
            assert not a[:, r].any()
        assert_same_bits(b[:, r], want[T // 2:, r], "following full call, " + name)


@pytest.mark.gpu
def test_gpu_voice_bank_matches_reference_golden_and_row_mask(gpu):
    g = np.load(GOLD)
    ev = g["events"].view(wl.VOICE_EVENTS_DTYPE).reshape(g["shape"][0], g["shape"][1])
    V = ev.shape[1]
    vb = gpu.VoiceBank(float(g["sr"]), *wl.voice_bank_params(V), flags=wl.VOICES_MIDI)
    vb2 = gpu.VoiceBank(float(g["sr"]), *wl.voice_bank_params(V), flags=wl.VOICES_MIDI)
    try:
        got = vb.process_host(ev)
        part = vb2.process_host(ev, row_mask=0b00000011)  # pitch and gate only
    finally:
        vb.close()
        vb2.close()
    assert_same_bits(got, g["out"], "voice bank vs reference golden")
    assert_same_bits(part[:, :2], g["out"][:, :2], "row_mask planes")
    assert not part[:, 2:].any()


@pytest.mark.gpu
def test_voice_rows_feed_a_graph(gpu, port_bank, port):
    """The bank's out planes have the layout of graph inputs: pitch row -> (x 2^-7 as cycles/sample)
    -> SineGen -> x gate row.  Whole path on the device, checked against port(bank) -> port(graph)."""
    import torch
    from madronalib_b200.graph import GraphSpec, SINE_ZERO_PHASE
    V, T = 64, 20
    ev = wl.voice_events(V, T, seed=9)
    prm = wl.voice_bank_params(V)
    rows, _ = port_bank.run(48000.0, *prm, ev)
    g = GraphSpec()
    pitch, gate = g.input(0), g.input(1)
    k = g.param()
    y = g.node("MULTIPLY", g.node("SINE", g.node("MULTIPLY", pitch, k)), gate)
    g.output(y)
    coef, state = g.new_coefs(V), g.new_state(V)
    coef[0] = np.float32(2.0 ** -7)
    state[0] = SINE_ZERO_PHASE
    inp = np.ascontiguousarray(rows[:, 0:2])
    want, _, _ = port.run(g, V, T, inp, state, coef)
    dev = torch.device("cuda", 0)
    d_ev = torch.from_numpy(ev.view(np.uint8).reshape(T, V, 72).copy()).to(dev)
    d_rows = torch.zeros((T, 8, V, 64), dtype=torch.float32, device=dev)
    vb = gpu.VoiceBank(48000.0, *prm)
    vg = gpu.VoiceGraph(g, V)
    try:
        sh = torch.cuda.current_stream().cuda_stream
        vb.process_device(d_ev, d_rows, T, 0xFF, sh)
        d_in = d_rows[:, 0:2].contiguous()
        d_out = torch.empty((T, 1, V, 64), dtype=torch.float32, device=dev)
        vg.set_coefs(coef)
        vg.set_state(state)
        vg.process_device(d_in, d_out, None, T, sh)
        torch.cuda.synchronize()
        got = d_out.cpu().numpy()
        # the same without the slicing copy: the graph is told that its input buffer has 8 planes per block
        vg.set_state(state)
        vg.set_input_planes(8)
        d_out2 = torch.empty_like(d_out)
        vg.process_device(d_rows, d_out2, None, T, sh)
        torch.cuda.synchronize()
        got2 = d_out2.cpu().numpy()
    finally:
        vb.close()
        vg.close()
    assert_same_bits(got, want, "events -> voice rows -> graph")
    assert_same_bits(got2, want, "events -> voice rows -> graph, 8-plane input buffer")


@pytest.mark.parametrize("mpe,unison,polyphony", [(False, False, 4), (False, True, 3), (True, False, 6)])
def test_router_c_abi_plus_port_bank_equals_reference(ref_bank, port_bank, mpe, unison, polyphony):
    """The C face of the router (mlb_router_*, host only) -> records -> Voice bank (the C port here) against
    the complete reference EventsToSignals, driven from Python with a seeded phrase."""
    from madronalib_b200 import api
    sr, glide, drift, T, P = 48000.0, 0.02, 0.5, 150, polyphony
    rng = np.random.default_rng(21 + polyphony)
    router = api.EventRouter(P, api.EventRouter.MPE if mpe else api.EventRouter.MIDI, unison=unison)
    held, phrase = [], []
    for t in range(T):
        base = t * 64
        evs = []
        if rng.random() < 0.3:
            key = int(rng.integers(40, 80))
            chan = int(rng.integers(2, 10)) if mpe else 1
            evs.append((api.EventRouter.NOTE_ON, chan, key, base + int(rng.integers(64)), key / 12.0, float(rng.random() * 0.8 + 0.2)))
            held.append((chan, key))
        if held and rng.random() < 0.25:
            chan, key = held.pop(int(rng.integers(len(held))))
            evs.append((api.EventRouter.NOTE_OFF, chan, key, base + int(rng.integers(64)), 0.0, 0.0))
        if rng.random() < 0.2:
            evs.append((api.EventRouter.PITCH_BEND, int(rng.integers(1, 10)), 0, base + int(rng.integers(64)), float(rng.random() * 2 - 1), 0.0))
        if rng.random() < 0.2:
            evs.append((api.EventRouter.CHANNEL_PRESSURE, int(rng.integers(1, 10)), 0, base + int(rng.integers(64)), float(rng.random()), 0.0))
        if rng.random() < 0.15:
            evs.append((api.EventRouter.CONTROLLER, int(rng.integers(1, 10)), int(rng.choice([16, 73, 74])), base + int(rng.integers(64)), float(rng.random()), 0.0))
        if rng.random() < 0.08:
            evs.append((api.EventRouter.SUSTAIN_PEDAL, 1, 0, base + int(rng.integers(64)), float(rng.integers(2)), 0.0))
        for e in evs:
            phrase.append(e)
            router.add_event(*e)
    NR = router.n_records
    recs = np.zeros((T, NR), wl.VOICE_EVENTS_DTYPE)
    for t in range(T):
        assert router.process_vector(t * 64, recs[t]) == 0
    router.close()
    first = 1 if mpe else 0
    idx = np.arange(NR, dtype=np.int32) + (0 if mpe else 1)
    bend = np.full(NR, 24.0 if mpe else 7.0, np.float32)
    if mpe:
        bend[0] = 7.0
    # the port bank: MPE main-voice rows are added by a post-pass (mlport_bank_set_main_voices)
    import ctypes
    L = port_bank.lib
    L.mlport_bank_create.restype = ctypes.c_void_p
    gs, da = np.full(NR, glide, np.float32), np.full(NR, drift, np.float32)
    h = L.mlport_bank_create(NR, ctypes.c_float(sr), idx.ctypes.data_as(ctypes.c_void_p), gs.ctypes.data_as(ctypes.c_void_p),
                             da.ctypes.data_as(ctypes.c_void_p), bend.ctypes.data_as(ctypes.c_void_p), 0 if mpe else 1)
    if mpe:
        mainv = np.full(NR, 0, np.int32)
        mainv[0] = -1
        L.mlport_bank_set_main_voices.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.mlport_bank_set_main_voices(h, mainv.ctypes.data_as(ctypes.c_void_p))
    got = np.zeros((T, 8, NR, 64), np.float32)
    L.mlport_bank_process.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    L.mlport_bank_process.restype = ctypes.c_double
    L.mlport_bank_process(h, T, recs.ctypes.data_as(ctypes.c_void_p), got.ctypes.data_as(ctypes.c_void_p), 1)
    L.mlport_bank_destroy.argtypes = [ctypes.c_void_p]
    L.mlport_bank_destroy(h)
    got = np.ascontiguousarray(got[:, :, first:, :].transpose(0, 2, 1, 3))  # -> [T][P][8][64]
    assert_events_to_signals(got, lambda: _reference_events_to_signals(sr, P, glide, drift, unison, mpe, T, phrase),
                             sr, P, glide, drift, unison, mpe, T, phrase)
    assert got[:, :, 1].max() > 0.1  # gates happened


def _reference_events_to_signals(sr, P, glide, drift, unison, mpe, T, phrase):
    """The complete reference EventsToSignals on `phrase` -> [T][P][8][64]."""
    from oracle.bindings import RefEventsToSignals
    ref = RefEventsToSignals(sr, P, glide, drift, unison=unison, mpe=mpe)
    for e in phrase:
        ref.add_event(*e)
    want = np.zeros((T, P, 8, 64), np.float32)
    for t in range(T):
        want[t] = ref.process_vector(t * 64)
    ref.close()
    return want


# ---- fuzz: random phrases, polyphony 1..16, MIDI / unison / MPE, several sample rates, against the complete
# reference EventsToSignals (CPU only; the bank is the C port) ----
def _fuzz_imports():
    import ctypes
    from madronalib_b200 import api
    return ctypes, api


def _router_fuzz_case(seed, PB):
    ctypes, api = _fuzz_imports()
    rng=np.random.default_rng(seed)
    mpe=bool(rng.integers(2)); unison=bool(rng.integers(2)) and not mpe
    P=int(rng.integers(1,17)); sr=float(rng.choice([44100.0,48000.0,96000.0])); glide=float(rng.choice([0.0,0.01,0.05])); drift=float(rng.choice([0.0,1.0]))
    T=int(rng.integers(40,200))
    dens=float(rng.choice([0.1,0.4,0.9]))
    router=api.EventRouter(P, 1 if mpe else 0, unison=unison)
    held, phrase=[], []
    E=api.EventRouter
    for t in range(T):
        base=t*64
        n=int(rng.poisson(dens))
        for _ in range(n):
            kind=int(rng.integers(8))
            tm=base+int(rng.integers(64))
            chan=int(rng.integers(1,11))
            if kind<=2:
                key=int(rng.integers(30,100)); ch=chan if mpe else 1
                e=(E.NOTE_ON,ch,key,tm,key/12.0,float(rng.random()*0.9+0.1)); held.append((ch,key))
            elif kind==3 and held:
                ch,key=held.pop(int(rng.integers(len(held)))); e=(E.NOTE_OFF,ch,key,tm,0.0,0.0)
            elif kind==4: e=(E.PITCH_BEND,chan,0,tm,float(rng.random()*2-1),0.0)
            elif kind==5: e=(E.CHANNEL_PRESSURE,chan,0,tm,float(rng.random()),0.0)
            elif kind==6: e=(E.CONTROLLER,chan,int(rng.choice([16,73,74,1,123,128,200])),tm,float(rng.choice([0.0,rng.random()])),0.0)
            elif kind==7: e=(int(rng.choice([E.SUSTAIN_PEDAL,E.NOTE_PRESSURE])),chan,int(rng.integers(30,100)),tm,float(rng.random()),0.0)
            else: continue
            phrase.append(e); router.add_event(*e)
    NR=router.n_records
    recs=np.zeros((T,NR),wl.VOICE_EVENTS_DTYPE)
    over=0
    for t in range(T):
        over+=router.process_vector(t*64,recs[t])
    router.close()
    if over: return "overflow(%d)"%over
    first=1 if mpe else 0
    idx=np.arange(NR,dtype=np.int32)+(0 if mpe else 1)
    bend=np.full(NR,24.0 if mpe else 7.0,np.float32)
    if mpe: bend[0]=7.0
    L=PB.lib
    gs,da=np.full(NR,glide,np.float32),np.full(NR,drift,np.float32)
    h=L.mlport_bank_create(NR,ctypes.c_float(sr),idx.ctypes.data_as(ctypes.c_void_p),gs.ctypes.data_as(ctypes.c_void_p),da.ctypes.data_as(ctypes.c_void_p),bend.ctypes.data_as(ctypes.c_void_p),0 if mpe else 1)
    if mpe:
        mainv=np.full(NR,0,np.int32); mainv[0]=-1
        L.mlport_bank_set_main_voices.argtypes=[ctypes.c_void_p,ctypes.c_void_p]; L.mlport_bank_set_main_voices(h,mainv.ctypes.data_as(ctypes.c_void_p))
    got=np.zeros((T,8,NR,64),np.float32)
    L.mlport_bank_process(h,T,recs.ctypes.data_as(ctypes.c_void_p),got.ctypes.data_as(ctypes.c_void_p),1)
    L.mlport_bank_destroy.argtypes=[ctypes.c_void_p]; L.mlport_bank_destroy(h)
    got=np.ascontiguousarray(got[:,:,first:,:].transpose(0,2,1,3))
    assert_events_to_signals(got, lambda: _reference_events_to_signals(sr, P, glide, drift, unison, mpe, T, phrase),
                             sr, P, glide, drift, unison, mpe, T, phrase)
    return "ok"


@pytest.mark.parametrize("seed", range(24))
def test_router_fuzz_against_reference(ref_bank, port_bank, seed):
    r = _router_fuzz_case(seed, port_bank)
    assert r == "ok" or r.startswith("overflow"), r

"""The compiled reference's answers, recorded where oracle/_ref exists and replayed everywhere else.

The tests compare against the reference itself (oracle/_ref: madronalib compiled in place), which only a
machine with the reference sources can build.  Every call a test makes on it is identified by a digest of
the method and its arguments; what it returned is kept in tests/golden/reference.npz:

* results the C port (oracle/_port) can compute as well -- graph runs, coefficient design, the Voice bank,
  the resampler banks -- are kept as the SHA-256 of their words (scalars as their values).  Replaying such a
  call runs the port with the same arguments, and the port's result must have the recorded digest or value:
  the test then works with words that are the reference's, bit for bit (float NaN payloads aside, as in
  tests/common.assert_same_bits).  Wall-clock seconds some calls also return are not compared.
* results only the reference computes (its own example bodies, FDN<SIZE> objects, wrappers) are kept whole.

A call that was never recorded fails.  Re-record after changing what a test asks the reference, with the whole
suite on a GPU machine where oracle/_ref is built (the device tests consult the reference too).  The file named
receives exactly the calls made in that session:

    MLB_RECORD_REFERENCE=tests/golden/reference.npz python -m pytest tests
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference.npz")
RECORDING = os.environ.get("MLB_RECORD_REFERENCE", "")

_store = None      # key -> list of encoded result items
_arrays = {}       # npz member name -> array kept whole
_dirty = False


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(GOLDEN) and not RECORDING:
            with np.load(GOLDEN) as z:
                _store = json.loads(bytes(z["index"]).decode())
                _arrays.update({k: z[k] for k in z.files if k != "index"})
    return _store


def save():
    """Write the recorded results (only after a recording run)."""
    if not _dirty:
        return
    index = np.frombuffer(json.dumps(_store, sort_keys=True).encode(), np.uint8)
    np.savez_compressed(RECORDING, index=index, **_arrays)


def _feed(h, x):
    from madronalib_b200.graph import GraphSpec
    if isinstance(x, GraphSpec):
        h.update(repr(("GraphSpec", [int(v) for v in x.ops], [tuple(int(i) for i in t) for t in x.ins],
                       [int(v) for v in x.iargs], [int(v) for v in x.outs])).encode())
    elif isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        h.update(repr(("ndarray", a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(("(%d" % len(x)).encode())
        for v in x:
            _feed(h, v)
        h.update(b")")
    elif isinstance(x, dict):
        for k in sorted(x):
            _feed(h, (k, x[k]))
    elif isinstance(x, np.generic):
        _feed(h, x.item())
    else:
        h.update(repr((type(x).__name__, x)).encode())


def _key(*parts) -> str:
    h = hashlib.sha256()
    _feed(h, parts)
    return h.hexdigest()[:32]


def digest(a: np.ndarray) -> str:
    """SHA-256 of an array's words, every NaN of a float32 array written as one canonical NaN."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(repr((a.dtype.str, a.shape)).encode())
    if a.dtype == np.float32:
        w = a.view(np.uint32).copy()
        w[np.isnan(a)] = 0x7FC00000
        a = w
    h.update(a.tobytes())
    return h.hexdigest()


def _items(res):
    return (list(res), True) if isinstance(res, tuple) else ([res], False)


def _record(key, res, whole):
    global _dirty
    items, _ = _items(res)
    enc = []
    for i, v in enumerate(items):
        if isinstance(v, np.ndarray):
            if whole:
                _arrays["%s_%d" % (key, i)] = v
                enc.append({"array": "%s_%d" % (key, i)})
            else:
                enc.append({"digest": digest(v)})
        elif v is None or isinstance(v, (bool, int, float, str)):
            enc.append({"value": v})
        else:
            raise TypeError("cannot record a %s" % type(v).__name__)
    _load()[key] = enc
    _dirty = True


def _entry(key, what):
    enc = _load().get(key)
    if enc is None:
        raise LookupError("no recorded reference result for %s (key %s): re-record tests/golden/reference.npz "
                          "where oracle/_ref is built (see tests/recorded_reference.py)" % (what, key))
    return enc


class _Replay:
    """Stands for a reference object: `real()` builds it (recording only), `standin` is the port's equivalent
    (None where the port has none).  Stateful objects chain every call into the key of the next.  `timed`
    names the methods whose float results are wall-clock seconds."""

    def __init__(self, scope, real, standin, stateful=False, timed=()):
        self._scope, self._real, self._standin, self._stateful = scope, real, standin, stateful
        self._timed = timed
        self._obj = real() if RECORDING else None

    def close(self):
        for o in (self._obj, self._standin):
            if o is not None and hasattr(o, "close"):
                o.close()

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        what = "%s.%s" % (self._scope if isinstance(self._scope, str) else self._scope[0], name)

        def call(*args, **kw):
            # the thread count a checker runs on does not change its result, and differs between machines
            key = _key(self._scope, name, args, {k: v for k, v in kw.items() if k != "nthreads"})
            if self._stateful:
                self._scope = key
            by_port = self._standin is not None and hasattr(self._standin, name)
            if RECORDING:
                res = getattr(self._obj, name)(*args, **kw)
                _record(key, res, whole=not by_port)
                if by_port:
                    getattr(self._standin, name)(*args, **kw)  # keep a stateful stand-in in step
                return res
            enc = _entry(key, what)
            if by_port:
                res = getattr(self._standin, name)(*args, **kw)
                items, _ = _items(res)
                assert len(items) == len(enc), what
                for i, (v, e) in enumerate(zip(items, enc)):
                    if "digest" in e:
                        same = isinstance(v, np.ndarray) and digest(v) == e["digest"]
                    elif isinstance(v, float) and name in self._timed:
                        continue
                    elif isinstance(v, float) and isinstance(e["value"], float):
                        same = np.float32(v).view(np.uint32) == np.float32(e["value"]).view(np.uint32)
                    else:
                        same = v == e["value"]
                    assert same, "%s, result %d: the C port differs from the recorded reference" % (what, i)
                return res
            items = [(_arrays[e["array"]].copy() if "array" in e else e["value"]) for e in enc]
            return tuple(items) if len(items) > 1 else items[0]
        return call


def _port():
    from oracle import bindings
    if not os.path.exists(bindings.PORT_LIB):
        bindings.build("port")
    return bindings


def oracle():
    """The reference's graph oracle (bindings.RefOracle), recorded."""
    b = _port()
    return _Replay("RefOracle", b.RefOracle, b.PortOracle())


def voice_bank():
    """The reference's own EventsToSignals::Voice bank (bindings.ref_voice_bank), recorded."""
    b = _port()
    return _Replay("ref_voice_bank", b.ref_voice_bank, b.port_voice_bank(), timed=("run",))


def resampler(direction: int, octaves: int, n_voices: int):
    """The reference's Upsampler / Downsampler bank (bindings.Resampler("ref", ...)), recorded."""
    b = _port()
    return _Replay(("Resampler", direction, octaves, n_voices), lambda: b.Resampler("ref", direction, octaves, n_voices),
                   b.Resampler("port", direction, octaves, n_voices), stateful=True)


def assert_events_to_signals(got: np.ndarray, reference_run, *case):
    """`got` [T][polyphony][8][64] must be what the complete reference EventsToSignals computes for `case`
    (its arguments and event phrase); `reference_run()` computes that with bindings.RefEventsToSignals."""
    key = _key("RefEventsToSignals", case)
    if RECORDING:
        want = reference_run()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
        _record(key, want, whole=False)
        return
    assert digest(got) == _entry(key, "RefEventsToSignals")[0]["digest"], \
        "router + bank differ from the recorded reference EventsToSignals"

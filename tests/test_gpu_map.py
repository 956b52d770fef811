"""Stateless elementwise ops (every DEFINE_OP* of MLDSPOps.h) on the GPU vs the port oracle."""
import zlib

import numpy as np
import pytest

from madronalib_b200.graph import GraphSpec, OP_TABLE
from tests.common import assert_same_bits

pytestmark = pytest.mark.gpu

STATELESS = [n for n, (op, nin, nst, nco) in OP_TABLE.items() if 30 <= op < 100]  # MLB_OP_MAP_FIRST..END
# _mm_rcp_ps / _mm_rsqrt_ps are CPU-microarchitecture-defined 12-bit approximations
HW_APPROX = {"SQRT_APPROX": 1.5 * 2.0 ** -12, "DIVIDE_APPROX": 1.5 * 2.0 ** -12}

SPECIALS = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 1e38, -1e38, 3e9, -3e9,
                     2147483648.0, -2147483648.0, 0.5, 1.5, 2.5, -0.5, -1.5, 88.5, -88.5, 100, -100,
                     1.0, -1.0, np.pi, -np.pi, 8191.5, 1e-20], np.float32)


def make_inputs(nin, n_rows, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((nin, n_rows, 64)) * 4.0).astype(np.float32)
    for k in range(nin):
        flat = x[k].reshape(-1)
        idx = rng.choice(flat.size, SPECIALS.size, replace=False)
        flat[idx] = SPECIALS
    return x


@pytest.mark.parametrize("name", STATELESS)
def test_map_op(gpu, port, name):
    nin = OP_TABLE[name][1]
    n_rows = 37
    x = make_inputs(nin, n_rows, zlib.crc32(name.encode()) % 1000)  # the same inputs in every process
    g = GraphSpec()
    g.output(g.node(name, *[g.input(k) for k in range(nin)]))
    inp = np.ascontiguousarray(x[:, None].transpose(1, 0, 2, 3))  # [T=1][nin][V=n_rows][64]
    want, _, _ = port.run(g, n_rows, 1, inp, g.new_state(n_rows), g.new_coefs(n_rows))
    want = want[0, 0]
    got = gpu.map_host(name, x[0], x[1] if nin > 1 else None, x[2] if nin > 2 else None)
    if name in HW_APPROX:
        # rcpps/rsqrtps treat denormal operands as zero, and flush a denormal reciprocal (of |b| > 1 / FLT_MIN) to
        # zero; the GPU does neither: compare normal inputs
        tiny = np.finfo(np.float32).tiny
        normal = np.all((np.abs(x[:nin]) >= tiny) | (x[:nin] == 0) | ~np.isfinite(x[:nin]), axis=0)
        if name == "DIVIDE_APPROX":
            normal &= ~(np.abs(x[1]) > np.float32(1.0) / tiny)
        ok = np.isfinite(want) & np.isfinite(got) & normal
        rel = np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-30)
        assert rel.max() <= 2 * HW_APPROX[name]
        assert np.array_equal(np.isnan(got)[normal], np.isnan(want)[normal])
    else:
        assert_same_bits(got, want, name)


def test_reference_precision_assertions(gpu):
    """Reference Tests/dspOpsTest.cpp:77-106: precise < 2e-6, approx < 2e-4 vs libm on
    rangeClosed(-pi, pi) (64 points); log covers x in (0, pi] only (NaNs drop out)."""
    kPi = np.float32(3.1415926535897932384626433)
    interval = (kPi - (-kPi)) / np.float32(63.0)
    a = (np.arange(64, dtype=np.float32) * interval + (-kPi)).astype(np.float32)[None, :]
    for name, fn in (("sin", np.sin), ("cos", np.cos), ("log", np.log), ("exp", np.exp)):
        with np.errstate(invalid="ignore", divide="ignore"):
            native = fn(a.astype(np.float32)).astype(np.float32)
        precise = gpu.map_host(name, a)
        approx = gpu.map_host(name + "_approx", a)
        m = np.isfinite(native) & (a > 0 if name == "log" else True)
        assert np.abs(native[m] - precise[m]).max() < 2e-6, name
        assert np.abs(native[m] - approx[m]).max() < 2e-4, name


def test_reference_lerp_and_fractional_part(gpu):
    """Reference Tests/dspOpsTest.cpp:148-165."""
    a = np.arange(64, dtype=np.float32)[None, :]
    b = np.zeros_like(a)
    c = gpu.map_host("lerp", a, b, np.full_like(a, 0.5))
    assert c[0, 63] == 63 * 0.5
    fa = gpu.map_host("fractional_part", np.full((1, 64), 1.25, np.float32))
    fb = gpu.map_host("fractional_part", np.full((1, 64), -1.25, np.float32))
    assert fa[0, 63] == -fb[0, 63] == 0.25

"""SURVEY 8(f) row 4: Upsampler / Downsampler banks (MLDSPFilters.h:1316-1473).  CPU: the C port against the
reference's own classes, with different call splits (filter states, buffers and the write counter carry
over).  GPU: the CUDA bank through the C ABI against the port, bit for bit."""
import numpy as np
import pytest

from tests.common import assert_same_bits


def _signal(T, V, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((T, V, 64)).astype(np.float32)


@pytest.mark.parametrize("direction", [0, 1])
@pytest.mark.parametrize("octaves", [1, 2, 3, 4])
def test_port_equals_reference_resamplers(ref, direction, octaves):
    from oracle.bindings import Resampler
    from tests import recorded_reference
    V = 9
    x = _signal(37, V, 5 + octaves)
    a, b = recorded_reference.resampler(direction, octaves, V), Resampler("port", direction, octaves, V)
    ya = np.concatenate([a.process(x[:10]), a.process(x[10:])])
    yb = np.concatenate([b.process(x[:10]), b.process(x[10:23]), b.process(x[23:])])
    a.close(), b.close()
    assert ya.shape == yb.shape == ((37 << octaves, V, 64) if direction == 0 else (37 >> octaves, V, 64))
    assert np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    assert np.abs(ya).max() > 0.1


@pytest.mark.gpu
@pytest.mark.parametrize("direction", [0, 1])
@pytest.mark.parametrize("octaves,V", [(1, 40), (2, 129), (3, 33), (4, 7)])
def test_gpu_resampler_bit_exact(gpu, port, direction, octaves, V):
    from oracle.bindings import Resampler
    x = _signal(41, V, 50 + octaves + direction)
    p = Resampler("port", direction, octaves, V)
    want = p.process(x)
    p.close()
    g = gpu.ResamplerBank(direction, octaves, V)
    try:
        got = np.concatenate([g.process_host(x[:5]), g.process_host(x[5:18]), g.process_host(x[18:])])
        g.clear()
        again = g.process_host(x)
    finally:
        g.close()
    assert_same_bits(got, want, "resampler, split calls")
    assert_same_bits(again, want, "resampler after clear()")


@pytest.mark.gpu
def test_gpu_up_then_down_is_a_delayed_copy(gpu):
    """Sanity on the signal level: 2x up then 2x down returns the input, low-passed and delayed a few samples."""
    V = 8
    n = np.arange(64 * 40, dtype=np.float32)
    x = np.sin(2 * np.pi * 0.01 * n).astype(np.float32).reshape(40, 1, 64).repeat(V, axis=1)
    up, down = gpu.ResamplerBank(0, 1, V), gpu.ResamplerBank(1, 1, V)
    try:
        y = down.process_host(up.process_host(x))
    finally:
        up.close(), down.close()
    a, b = x[:, 0].reshape(-1), y[:, 0].reshape(-1)
    best = max(abs(np.corrcoef(a[200:2000], b[200 + d:2000 + d])[0, 1]) for d in range(0, 12))
    assert best > 0.999

"""GPU parity of the coefficient-ROW (modulated / swept) filter forms against the reference's own
operator()(vx, omega, k) / operator()(vx, vc) (MLDSPFilters.h:136-152,304-319,385-400)."""
import numpy as np
import pytest

from madronalib_b200 import workloads as wl
from tests.common import assert_same_bits, assert_state_equal, run_gpu

pytestmark = pytest.mark.gpu

EXACT_CASES = [c for c in wl.SWEPT_CASES if c != "lopass_mod"]


@pytest.mark.parametrize("name", EXACT_CASES)
@pytest.mark.parametrize("n_voices,n_blocks,splits", [(37, 7, (3, 4)), (200, 5, None)])
def test_swept_filters_bit_exact(gpu, port, ref, name, n_voices, n_blocks, splits):
    w = wl.swept_filter_case(name, n_voices, n_blocks)
    inp = w.inputs(n_blocks)
    ro, _, rs = ref.run(w.spec, n_voices, n_blocks, inp, w.state, w.coef)
    _, pm, _ = port.run(w.spec, n_voices, n_blocks, inp, w.state, w.coef, want_mix=True, mix_mode=1)
    fused_expected = name in ("lopass_v", "sine_lopass_v_gain")
    for flags in ((0, gpu.FLAG_FORCE_GENERIC) if fused_expected else (0,)):
        go, gm, gs, kname = run_gpu(gpu, w, n_blocks, inp, flags=flags, want_mix=True, splits=splits)
        assert kname.startswith("fused:") == (fused_expected and flags == 0), kname
        assert_same_bits(go, ro, name + " out " + kname)
        assert_same_bits(gm, pm, name + " mix " + kname)
        assert_state_equal(gs, rs, name + " state " + kname)


def test_lopass_v_equals_the_reference_operator_itself(gpu, ref):
    """One voice, omega / k sweeps with the clamp canaries: host makeCoeffsVec rows + device LOPASS_V
    == Lopass::operator()(vx, omega, k) called directly in the compiled reference."""
    T = 9
    rng = np.random.default_rng(4)
    n = np.arange(T * 64, dtype=np.float32).reshape(T, 1, 64)
    omega = (0.02 + 0.3 * (0.5 + 0.5 * np.sin(n * 0.013))).astype(np.float32)
    omega[0, 0, :4] = [0.6, 0.5, 0.499, 0.0]
    k = (0.005 + 1.5 * rng.random((T, 1, 64))).astype(np.float32)
    x = (rng.standard_normal((T, 1, 64)) * 0.5).astype(np.float32)
    want = ref.lopass_mod(x[:, 0], omega[:, 0], k[:, 0])
    w = wl.swept_filter_case("lopass_v", 1, T, x=x, omega=omega, k=k)
    go, _, _, kname = run_gpu(gpu, w, T, w.inputs(T))
    assert kname.startswith("fused:"), kname
    assert_same_bits(go[:, 0, 0], want, "LOPASS_V vs Lopass::operator()(vx, omega, k)")


def test_fused_swept_chain_large_bank_default_launch_shape(gpu, port, ref):
    """SineGen -> Lopass(coefficient rows) -> gain through the persistent multi-plane chain grid
    (20 000 voices > 4 * SMs groups: dynamic work units, state hopping), ragged last group, mix bus."""
    V, T = 20000 + 13, 16
    w = wl.swept_filter_case("sine_lopass_v_gain", V, T)
    inp = w.inputs(T)
    ro, _, rs = ref.run(w.spec, V, T, inp, w.state, w.coef, nthreads=16)
    _, pm, _ = port.run(w.spec, V, T, inp, w.state, w.coef, want_out=False, want_mix=True, mix_mode=1, nthreads=16)
    go, gm, gs, kname = run_gpu(gpu, w, T, inp, want_mix=True, splits=(9, 7))
    assert kname.startswith("fused:"), kname
    assert_same_bits(go, ro, "swept chain out")
    assert_same_bits(gm, pm, "swept chain mix")
    assert_state_equal(gs, rs, "swept chain state")


def test_lopass_mod_device_coefficients_within_tolerance(gpu, port, ref):
    """LOPASS_MOD designs the coefficients on the device (CUDA sinf, not glibc's): the approximate
    variant.  Stated tolerance (DESIGN.md 5): 2e-5 of the output's peak over 12 blocks of sweeps
    with k >= 0.05 (Q <= 20)."""
    V, T = 150, 12
    w = wl.swept_filter_case("lopass_mod", V, T)
    inp = w.inputs(T)
    ro, _, _ = ref.run(w.spec, V, T, inp, w.state, w.coef)
    go, _, _, kname = run_gpu(gpu, w, T, inp)
    err = float(np.abs(go - ro).max() / np.abs(ro).max())
    print("LOPASS_MOD max error relative to peak:", err, kname)
    assert err <= 2e-5

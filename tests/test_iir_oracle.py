"""CPU: the numpy restatement of the bank's IIR filters (tests/sxiir.py), which the GPU tests
compare the kernels against, is scipy.signal.sosfilt bit for bit on complex64 input with float32
coefficients -- outputs and final state, with a nonzero initial state and a zero tail that drives
the state into subnormals -- carries its state across blocks exactly, and is within a stated
tolerance of sosfilt in float64.  The ctypes bindings of the new entry points are checked without a
GPU."""
import re
from pathlib import Path

import numpy as np
import pytest

import sxiir

signal = pytest.importorskip("scipy.signal")

ROOT = Path(__file__).resolve().parent.parent

# Stable designs of 1 to 8 sections: low-pass, high-pass and band-pass.
DESIGNS = {
    "butter1": lambda: signal.butter(1, 0.2, output="sos"),
    "butter4_hp": lambda: signal.butter(4, 0.2, btype="highpass", output="sos"),
    "cheby1_6": lambda: signal.cheby1(6, 1.0, 0.25, output="sos"),
    "cheby2_6": lambda: signal.cheby2(6, 40.0, 0.25, output="sos"),
    "butter8": lambda: signal.butter(8, 0.1, output="sos"),
    "ellip10": lambda: signal.ellip(10, 0.5, 60.0, 0.3, output="sos"),
    "butter12_bp": lambda: signal.butter(6, [0.1, 0.3], btype="bandpass", output="sos"),
    "butter16": lambda: signal.butter(16, 0.3, output="sos"),
    "ellip8_bp": lambda: signal.ellip(8, 0.5, 60.0, [0.1, 0.3], btype="bandpass", output="sos"),
}

# float32 against float64 (coefficients and arithmetic), as a fraction of the output's peak:
# measured up to 7e-6 over these designs and inputs.
FLOAT64_TOLERANCE = 5e-5


def complex_input(rng, nstreams, n, tail=0):
    x = (rng.standard_normal((nstreams, n)) + 1j * rng.standard_normal((nstreams, n))).astype(np.complex64)
    x *= np.float32(0.3)
    if tail:
        x[:, -tail:] = 0
    x[0, : n // 4] = x[0, : n // 4].real  # an imaginary part of exactly zero
    return x


def initial_state(rng, nsections, nstreams):
    z = rng.standard_normal((nsections, nstreams, 2)) + 1j * rng.standard_normal((nsections, nstreams, 2))
    return (0.1 * z).astype(np.complex64)


@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_restatement_is_sosfilt_bit_for_bit(name):
    sos = DESIGNS[name]()
    assert 1 <= sos.shape[0] <= sxiir.MAX_SECTIONS
    rng = np.random.default_rng(sos.shape[0])
    x = complex_input(rng, 6, 2500, tail=2000)
    zi = initial_state(rng, sos.shape[0], 6)
    y, zf = sxiir.sosfilt(sos, x, zi)
    want_y, want_zf = signal.sosfilt(sxiir.sos32(sos), x, zi=zi)
    assert want_y.dtype == np.complex64
    assert np.array_equal(y.view(np.uint32), want_y.view(np.uint32))
    assert np.array_equal(zf.view(np.uint32), want_zf.view(np.uint32))
    # the zero tail has driven the state into subnormals, where both still agree
    f = np.abs(zf.view(np.float32))
    assert ((f > 0) & (f < np.finfo(np.float32).tiny)).any()


@pytest.mark.parametrize("name", ["butter1", "cheby2_6", "ellip8_bp"])
def test_blockwise_with_carried_state_equals_one_shot(name):
    sos = DESIGNS[name]()
    rng = np.random.default_rng(7)
    x = complex_input(rng, 5, 1000, tail=300)
    zi = initial_state(rng, sos.shape[0], 5)
    whole, zf = sxiir.sosfilt(sos, x, zi)
    parts, z = [], zi
    for a, b in zip([0, 1, 257, 600], [1, 257, 600, 1000]):
        y, z = sxiir.sosfilt(sos, x[:, a:b], z)
        parts.append(y)
    assert np.array_equal(np.concatenate(parts, axis=1).view(np.uint32), whole.view(np.uint32))
    assert np.array_equal(z.view(np.uint32), zf.view(np.uint32))


@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_restatement_is_close_to_float64(name):
    sos = DESIGNS[name]()
    x = complex_input(np.random.default_rng(3), 8, 4000)
    y, _ = sxiir.sosfilt(sos, x)
    want = signal.sosfilt(sos, x.astype(np.complex128))
    assert np.abs(y - want).max() <= FLOAT64_TOLERANCE * np.abs(want).max()


def test_filter_entry_points_have_bindings():
    from sxxcvr_b200 import capi
    header = (ROOT / "include" / "sxgpu.h").read_text()
    assert re.search(r"#define SXGPU_IIR_MAX_SECTIONS\s+(\d+)", header).group(1) == str(sxiir.MAX_SECTIONS)
    for name in ("sxgpu_iir_create", "sxgpu_iir_destroy", "sxgpu_iir_set_state", "sxgpu_iir_get_state",
                 "sxgpu_iir_apply", "sxgpu_bank_repeat_filtered", "sxgpu_iir_device_view"):
        assert name + "(" in header
        assert name in capi.SIGNATURES


def test_iir_rejects_a_malformed_sos_before_the_library():
    from sxxcvr_b200 import Iir
    ctx = type("Ctx", (), {"lib": None, "handle": None})()
    with pytest.raises(ValueError):
        Iir(ctx, 4, np.zeros(6))

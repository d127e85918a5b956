"""CPU: the numpy restatement of sxgpu_iir_apply_long (tests/sxiir_long.py), which the GPU tests
compare the kernels against bit for bit.  Its first chunk and a block of one chunk are the
sequential float32 filter (tests/sxiir.py, scipy's sosfilt on complex64) bit for bit; past the first
chunk it stays within the float32 filter's own tolerance of sosfilt in float64, and within a few
1e-6 of the peak of sosfilt in float32, over thousands of chunks with a nonzero initial state and a
short last chunk.  Its powers of the state matrix are the float64 recurrence on zero input."""
import numpy as np
import pytest

import sxiir
import sxiir_long
from test_iir_oracle import DESIGNS, FLOAT64_TOLERANCE, ROOT, complex_input, initial_state

signal = pytest.importorskip("scipy.signal")

# Against sosfilt on complex64 with the float32 coefficients, as a fraction of its peak: measured up
# to 8.6e-7 (ellip8_bp) over these designs and inputs, 1e-10 or less for the well-damped ones.
FLOAT32_TOLERANCE = 5e-6

# 2 streams of 4097 chunks of 128 frames, the last of 37 frames: the chunk rule's own choice.
NSTREAMS, NFRAMES = 2, 4096 * 128 + 37


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.fixture(scope="module")
def long_runs():
    runs = {}
    for name in sorted(DESIGNS):
        sos = DESIGNS[name]()
        rng = np.random.default_rng(sos.shape[0] + 100)
        x = complex_input(rng, NSTREAMS, NFRAMES)
        zi = initial_state(rng, sos.shape[0], NSTREAMS)
        runs[name] = (sos, x, zi, sxiir_long.apply_long(sos, x, zi))
    return runs


def test_chunk_rule():
    assert sxiir_long.chunk_len(NSTREAMS, NFRAMES) == 128
    assert sxiir_long.chunk_len(1, 1 << 27) == 1024
    assert sxiir_long.chunk_len(16, 1 << 23) == 1024
    assert sxiir_long.chunk_len(1, 1 << 22) == 128
    assert sxiir_long.chunk_len(65536, 1 << 20) == 1024
    assert sxiir_long.chunk_len(64, 1 << 20) == 1024
    assert sxiir_long.chunk_len(32, 1 << 20) == 512


@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_close_to_float64(long_runs, name):
    sos, x, zi, (y, _) = long_runs[name]
    want = signal.sosfilt(sos, x.astype(np.complex128), zi=zi.astype(np.complex128))[0]
    assert np.abs(y - want).max() <= FLOAT64_TOLERANCE * np.abs(want).max()


@pytest.mark.parametrize("name", sorted(DESIGNS))
def test_close_to_float32_and_first_chunk_bit_exact(long_runs, name):
    sos, x, zi, (y, zf) = long_runs[name]
    want, want_zf = signal.sosfilt(sxiir.sos32(sos), x, zi=zi)
    assert np.abs(y - want).max() <= FLOAT32_TOLERANCE * np.abs(want).max()
    assert np.abs(zf - want_zf).max() <= FLOAT32_TOLERANCE * np.abs(want).max()
    assert same_bits(y[:, :128], want[:, :128])
    assert not same_bits(y, want)  # later chunks start from a rounded state


@pytest.mark.parametrize("name", ["butter1", "cheby2_6", "ellip8_bp"])
def test_one_chunk_is_the_sequential_filter(name):
    sos = DESIGNS[name]()
    rng = np.random.default_rng(5)
    for nstreams, nframes in ((1, 1), (3, 128), (1, 100)):
        assert sxiir_long.chunk_len(nstreams, nframes) >= nframes
        x = complex_input(rng, nstreams, nframes)
        zi = initial_state(rng, sos.shape[0], nstreams)
        y, zf = sxiir_long.apply_long(sos, x, zi)
        want_y, want_zf = sxiir.sosfilt(sos, x, zi)
        assert same_bits(y, want_y) and same_bits(zf, want_zf)


@pytest.mark.parametrize("name", ["butter1", "butter8", "ellip8_bp", "butter16"])
def test_powers_are_the_float64_recurrence(name):
    sos = DESIGNS[name]()
    c = sxiir.sos32(sos).astype(np.float64)
    chain = sxiir_long.power_chain(sos, 11)
    n = 2 * c.shape[0]
    z0 = np.random.default_rng(1).standard_normal(n)
    z = z0.copy()
    peak = np.abs(z0).max()
    for steps in range(1 << 10):
        x = 0.0
        for q in range(c.shape[0]):
            b0, b1, b2, _, a1, a2 = c[q]
            y = b0 * x + z[2 * q]
            z[2 * q], z[2 * q + 1] = (b1 * x - a1 * y) + z[2 * q + 1], b2 * x - a2 * y
            x = y
        peak = max(peak, np.abs(z).max())
        done = steps + 1
        if done & (done - 1) == 0:  # A^(2^j) z0 after 2^j steps
            j = done.bit_length() - 1
            got = sxiir_long.matvec(chain[j], z0)
            assert np.abs(got - z).max() <= 1e-12 * peak, (j, np.abs(got - z).max() / peak)


def test_apply_long_has_bindings():
    from sxxcvr_b200 import capi
    header = (ROOT / "include" / "sxgpu.h").read_text()
    assert "sxgpu_iir_apply_long(" in header
    assert "sxgpu_iir_apply_long" in capi.SIGNATURES

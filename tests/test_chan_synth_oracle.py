"""CPU: the numpy restatement of sxgpu_chan_synth_* (tests/sxchansynth.py), which the GPU tests compare
the kernel against bit for bit, is the synthesis channelizer it claims to be: it is within float32
rounding of the float64 definition, any split into calls gives the bits of one call, its step 2 is
sxfir's interpolator on each residue column bit for bit, it matches sxfir + sxnco per channel summed
over the channels, a constant in one channel comes out as a tone at that channel's centre, the
analysis channelizer followed by it reconstructs the signal, and its twiddles are the oscillator's
coarse table.  And chan_synth_kernel in libsxgpu.so contains no fused multiply-add."""
import re

import numpy as np
import pytest

import sxchan
import sxchansynth
import sxfir
import sxnco
from test_fir_oracle import same_bits

signal = pytest.importorskip("scipy.signal")

TOLERANCE = 1e-6  # of M max|y| max_t sum_p |h[t + p D]|

SHAPES = [(16, 16, 256), (16, 8, 200), (8, 2, 31), (64, 32, 768), (4, 4, 3), (2, 1, 5), (2, 2, 64),
          (1024, 1024, 3000), (1024, 512, 700)]


def design(ntaps, m):
    return signal.firwin(ntaps, 1.0 / m) if ntaps > 1 else np.array([0.9])


def noise(rng, nstreams, m, n):
    y = rng.standard_normal((nstreams, m, n)) + 1j * rng.standard_normal((nstreams, m, n))
    return y.astype(np.complex64)


def phase_sum(h, d):
    """max_t sum_p |h[t + p D]| of h rounded to float32."""
    h = np.abs(np.asarray(h, np.float64).astype(np.float32).astype(np.float64))
    return max(h[t::d].sum() for t in range(min(d, h.size)))


@pytest.mark.parametrize("m,d,ntaps", SHAPES)
def test_restatement_is_within_rounding_of_the_definition(m, d, ntaps):
    rng = np.random.default_rng(m + d + ntaps)
    h = design(ntaps, m)
    nin = -(-ntaps // d) + 9 if m < 1024 else 5
    y = noise(rng, 2, m, nin)
    got = sxchansynth.Stream(h, m, d, 2).feed(y)
    want = sxchansynth.definition(h, y, m, d)
    assert got.shape == want.shape == (2, nin * d)
    scale = m * np.abs(y).max() * phase_sum(h, d)
    err = np.abs(got.astype(np.complex128) - want).max() / scale
    assert err < TOLERANCE, err


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 200), (8, 2, 31), (4, 4, 3), (2, 1, 5), (64, 32, 768)])
def test_any_split_equals_one_call(m, d, ntaps):
    """Calls of 1 frame, of fewer frames than the history, of lengths that are not multiples of
    M / D, and a start at a phase other than 0."""
    rng = np.random.default_rng(ntaps)
    h = design(ntaps, m)
    total = 200
    y = noise(rng, 3, m, total)
    start = (m // d) - 1
    whole = sxchansynth.Stream(h, m, d, 3)
    whole.set_state(None, start)
    want = whole.feed(y)
    for cuts in ([1, 6, 93, 100], [1] * 40 + [160], [ntaps // (3 * d) + 1] * 3 + [7, 1, 2, 3, 5, 8, 13], [199, 1]):
        st, parts, i = sxchansynth.Stream(h, m, d, 3), [], 0
        st.set_state(None, start)
        for k in cuts:
            k = min(k, total - i)
            if k == 0:
                break
            parts.append(st.feed(y[:, :, i:i + k]))
            i += k
        if i < total:
            parts.append(st.feed(y[:, :, i:]))
        assert same_bits(np.concatenate(parts, axis=1), want), cuts
        assert same_bits(st.hist, whole.hist) and st.phase == whole.phase


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 200), (8, 2, 31), (2, 1, 5), (64, 32, 768), (4, 4, 3)])
def test_step_two_is_the_fir_interpolator_on_each_residue_column(m, d, ntaps):
    rng = np.random.default_rng(ntaps + 7)
    h = design(ntaps, m)
    S, nin = 2, 60
    y = noise(rng, S, m, nin)
    got = sxchansynth.Stream(h, m, d, S).feed(y)
    frames = np.ascontiguousarray(y.transpose(0, 2, 1))
    yr, yi = sxchansynth.idft(frames.real, frames.imag, m)
    n = np.arange(nin * d)
    for c in range(m):
        col = np.empty((S, nin), np.complex64)
        col.real, col.imag = yr[:, :, c], yi[:, :, c]
        z = sxfir.Stream(h, d, 1, S).feed(col)
        assert same_bits(np.ascontiguousarray(got[:, n % m == c]), np.ascontiguousarray(z[:, n % m == c])), c


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 200), (8, 2, 31), (2, 1, 5), (64, 32, 768)])
def test_channels_are_the_interpolator_then_the_oscillator_summed(m, d, ntaps):
    """sxfir(h, D, 1) of each channel, then sxnco at +k/M from output frame 0, summed over the
    channels: the same stream, within tolerance, over two calls."""
    rng = np.random.default_rng(m * d + 3)
    h = design(ntaps, m)
    S = 2
    y = noise(rng, S, m, 90)
    syn = sxchansynth.Stream(h, m, d, S)
    got = np.concatenate([syn.feed(y[:, :, :37]), syn.feed(y[:, :, 37:])], axis=1)
    freqs = [k / m if k < m // 2 else (k - m) / m for k in range(m)]
    fir, nco = sxfir.Stream(h, d, 1, S * m), sxnco.Stream(S * m, np.tile(freqs, S))
    want = np.concatenate([nco.feed(fir.feed(y[:, :, a:b].reshape(S * m, -1))).reshape(S, m, -1).astype(np.complex128).sum(axis=1)
                           for a, b in ((0, 37), (37, 90))], axis=1)
    scale = m * np.abs(y).max() * phase_sum(h, d)
    assert np.abs(got.astype(np.complex128) - want).max() / scale < TOLERANCE


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (8, 4, 96), (64, 32, 768)])
def test_a_constant_in_one_channel_is_a_tone_at_its_centre(m, d, ntaps):
    h = design(ntaps, m)
    h32 = h.astype(np.float32).astype(np.float64)
    hp, nin = -(-ntaps // d), -(-ntaps // d) + 16
    n = np.arange(nin * d)
    gain = np.array([h32[t::d].sum() for t in range(d)])[n % d]
    for k in (0, 1, m // 2, m - 1):
        y = np.zeros((1, m, nin), np.complex64)
        y[0, k] = 1.0
        x = sxchansynth.Stream(h, m, d, 1).feed(y)[0].astype(np.complex128)
        want = gain * np.exp(2j * np.pi * k * (n % m) / m)
        steady = slice((hp - 1) * d, None)
        assert np.abs(x[steady] - want[steady]).max() < 1e-5 * np.abs(h32).sum(), k


@pytest.mark.parametrize("m,d,na,ns", [(16, 8, 257, 129), (16, 8, 513, 129), (8, 4, 129, 65)])
def test_analysis_then_synthesis_reconstructs_the_signal(m, d, na, ns):
    """sxchan with firwin(na, 1/M), then this with firwin(ns, 2/M), oversampled by 2: x delayed by the
    two linear-phase delays (a multiple of M), scaled by a gain g within 0.5 % of 1 / D, with the
    error at least 50 dB below the signal after the start-up.  (g - 1/D is the prototypes' passband
    gain through the bank, 0.3 to 0.4 % here; it is a scale, not a distortion.)"""
    rng = np.random.default_rng(na + ns)
    delay = (na - 1) // 2 + (ns - 1) // 2
    assert delay % m == 0
    x = (rng.standard_normal((1, 8192)) + 1j * rng.standard_normal((1, 8192))).astype(np.complex64)
    y = sxchan.Stream(signal.firwin(na, 1.0 / m), m, d, 1).feed(x)
    xr = sxchansynth.Stream(signal.firwin(ns, 2.0 / m), m, d, 1).feed(y)[0].astype(np.complex128)
    start = na + ns
    ref = x[0, start:x.shape[1] - delay].astype(np.complex128)
    got = xr[delay + start:]
    g = np.vdot(ref, got) / np.vdot(ref, ref)
    assert abs(g * d - 1) < 5e-3, g
    err = got - g * ref
    snr = 10 * np.log10(np.mean(np.abs(g * ref) ** 2) / np.mean(np.abs(err) ** 2))
    assert snr > 50, snr


def test_twiddles_are_the_oscillator_table():
    for m in (2, 4, 16, 1024):
        tr, ti = sxchansynth.twiddles(m)
        q = np.arange(m // 2) * (1024 // m)
        assert same_bits(tr, sxnco.A_RE[q]) and same_bits(ti, sxnco.A_IM[q])
        assert tr.dtype == np.float32 and ti.dtype == np.float32
    tr, ti = sxchansynth.twiddles(1024)
    assert tr[0] == 1.0 and ti[0] == 0.0 and not np.signbit(ti[0])
    assert ti[256] == 1.0


def test_chan_synth_kernel_has_no_fused_multiply_add():
    import subprocess

    from sxxcvr_b200 import capi
    out = subprocess.run(["cuobjdump", "-sass", str(capi.library_path())], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump not available")
    kernels, name = {}, None
    for line in out.stdout.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            kernels[name] = []
        elif name:
            kernels[name].append(line)
    kernels = {k: "\n".join(v) for k, v in kernels.items() if "chan_synth_kernel" in k}
    assert kernels, "chan_synth_kernel is missing"
    for name, sass in kernels.items():
        assert not re.search(r"\bFFMA2?\b", sass), name
        assert re.search(r"\bFMUL2?\b", sass) and re.search(r"\bFADD2?\b", sass), name

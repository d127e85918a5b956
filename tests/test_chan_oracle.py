"""CPU: the numpy restatement of sxgpu_chan_* (tests/sxchan.py), which the GPU tests compare the
kernel against bit for bit, is the channelizer it claims to be: it is within float32 rounding of the
float64 definition, any split into calls gives the bits of one call, channel k is the oscillator at
-k/M followed by the FIR decimator, a tone at a channel's centre leaves every channel with the
prototype's response at their distance, and its twiddles are the oscillator's coarse table
conjugated.  And chan_apply_kernel in libsxgpu.so contains no fused multiply-add."""
import math
import re

import numpy as np
import pytest

import sxchan
import sxfir
import sxnco
from test_fir_oracle import same_bits

signal = pytest.importorskip("scipy.signal")

TOLERANCE = 1e-6  # of sum |h| max |x|

SHAPES = [(16, 16, 256), (16, 8, 200), (8, 2, 31), (64, 32, 768), (4, 4, 3), (2, 1, 5), (2, 2, 64),
          (1024, 1024, 3000), (1024, 512, 700)]


def design(ntaps, m):
    return signal.firwin(ntaps, 1.0 / m) if ntaps > 1 else np.array([0.9])


def noise(rng, nstreams, n):
    return (rng.standard_normal((nstreams, n)) + 1j * rng.standard_normal((nstreams, n))).astype(np.complex64)


@pytest.mark.parametrize("m,d,ntaps", SHAPES)
def test_restatement_is_within_rounding_of_the_definition(m, d, ntaps):
    rng = np.random.default_rng(m + d + ntaps)
    h = design(ntaps, m)
    x = noise(rng, 2, 2 * m + 3 * ntaps + 5 if m < 1024 else 4 * m + 7)
    got = sxchan.Stream(h, m, d, 2).feed(x)
    want = sxchan.definition(h, x, m, d)
    assert got.shape == want.shape
    scale = np.abs(h.astype(np.float32)).sum() * np.abs(x).max()
    err = np.abs(got.astype(np.complex128) - want).max() / scale
    assert err < TOLERANCE, err


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 200), (8, 2, 31), (4, 4, 3), (2, 1, 5), (64, 32, 768)])
def test_any_split_equals_one_call(m, d, ntaps):
    """Calls of 1 frame, of fewer frames than the history, and of lengths that are not multiples of D or M."""
    rng = np.random.default_rng(ntaps)
    h = design(ntaps, m)
    x = noise(rng, 3, 1000)
    whole = sxchan.Stream(h, m, d, 3)
    want = whole.feed(x)
    for cuts in ([1, 6, 493, 500], [1] * 40 + [960], [ntaps // 3 + 1] * 3 + [7, 1, 2, 3, 5, 8, 13], [999, 1]):
        st, parts, i = sxchan.Stream(h, m, d, 3), [], 0
        for k in cuts:
            k = min(k, 1000 - i)
            if k == 0:
                break
            parts.append(st.feed(x[:, i:i + k]))
            i += k
        if i < 1000:
            parts.append(st.feed(x[:, i:]))
        assert same_bits(np.concatenate(parts, axis=2), want), cuts
        assert same_bits(st.hist, whole.hist) and st.phase == whole.phase


def test_phase_and_output_counts():
    st = sxchan.Stream(design(31, 8), 8, 2)
    fed, total = 0, 0
    for n in (1, 1, 3, 8, 5, 100):
        want = sxchan.output_frames(fed, n, 2)
        assert st.feed(np.ones((1, n), np.complex64)).shape == (1, 8, want)
        fed += n
        total += want
        assert st.phase == fed % 8
    assert total == -(-fed // 2)


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (16, 8, 200), (8, 2, 31), (2, 1, 5), (64, 32, 768)])
def test_channel_k_is_the_oscillator_then_the_decimator(m, d, ntaps):
    """sxnco at -k/M with its phase set to X inc, then sxfir(h, 1, D): the same channel, within tolerance."""
    rng = np.random.default_rng(m * d)
    h = design(ntaps, m)
    x = noise(rng, 1, 700)
    ch = sxchan.Stream(h, m, d, 1)
    y = np.concatenate([ch.feed(x[:, :333]), ch.feed(x[:, 333:])], axis=2)[0]
    scale = np.abs(h.astype(np.float32)).sum() * np.abs(x).max()
    for k in range(m):
        f = -k / m
        f = f + 1.0 if f < -0.5 else f
        nco, fir = sxnco.Stream(1, [f]), sxfir.Stream(h, 1, d, 1)
        want = []
        for part in (x[:, :333], x[:, 333:]):
            nco.phase = ((fir.fed * nco.inc.astype(np.uint64)) % 2**32).astype(np.uint32)
            want.append(fir.feed(nco.feed(part)))
        want = np.concatenate(want, axis=1)[0]
        assert want.shape == y[k].shape
        assert np.abs(y[k].astype(np.complex128) - want).max() / scale < TOLERANCE, k


@pytest.mark.parametrize("m,d,ntaps", [(16, 16, 256), (8, 4, 96), (64, 32, 768)])
def test_a_tone_at_a_channel_centre_gives_the_prototype_response(m, d, ntaps):
    h = design(ntaps, m)
    h32 = h.astype(np.float32).astype(np.float64)
    n = ntaps + 64 * d
    for j in (0, 1, m // 2, m - 1):
        x = np.exp(2j * np.pi * j * np.arange(n) / m).astype(np.complex64)[None]
        y = sxchan.Stream(h, m, d, 1).feed(x)[0]
        steady = y[:, -(-ntaps // d):]
        _, resp = signal.freqz(h32, worN=2 * np.pi * ((j - np.arange(m)) / m))
        assert np.abs(np.abs(steady) - np.abs(resp)[:, None]).max() < 1e-5 * np.abs(h32).sum(), j
    # the passband of the centre channel, and a channel two away in the stopband
    assert abs(abs(resp[j]) - 1.0) < 1e-2 and abs(resp[(j + 2) % m]) < 1e-2


def test_twiddles_are_the_oscillator_table_conjugated():
    for m in (2, 4, 16, 1024):
        tr, ti = sxchan.twiddles(m)
        q = np.arange(m // 2) * (1024 // m)
        assert same_bits(tr, sxnco.A_RE[q]) and same_bits(ti, -sxnco.A_IM[q])
        assert tr.dtype == np.float32 and ti.dtype == np.float32
    tr, ti = sxchan.twiddles(1024)
    assert tr[0] == 1.0 and math.copysign(1.0, float(ti[0])) == -1.0  # T[0].im is -0
    assert ti[256] == -1.0 and tr[256] == np.float32(math.cos(math.pi / 2))


def chan_kernel_sass():
    from sxxcvr_b200 import capi
    import subprocess
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
    return {k: "\n".join(v) for k, v in kernels.items() if "chan_apply_kernel" in k}


def test_chan_kernel_has_no_fused_multiply_add():
    kernels = chan_kernel_sass()
    assert kernels, "chan_apply_kernel is missing"
    for name, sass in kernels.items():
        assert not re.search(r"\bFFMA2?\b", sass), name
        assert re.search(r"\bFMUL2?\b", sass) and re.search(r"\bFADD2?\b", sass), name

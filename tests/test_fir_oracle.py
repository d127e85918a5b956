"""CPU: the numpy restatement of sxgpu_fir_apply (tests/sxfir.py), which the GPU tests compare the
kernels against bit for bit, equals scipy.signal.upfirdn on each stream's concatenated input bit
for bit, over random splits of the input into calls; and the FIR kernels in libsxgpu.so contain no
fused multiply-add, which would change the bits."""
import re
import subprocess

import numpy as np
import pytest

import sxfir

signal = pytest.importorskip("scipy.signal")

# (ntaps, up, down): 1 tap, ntaps < up, ntaps not a multiple of up, up == down > 1, coprime and
# non-coprime factors, the shapes of the GPU tests and the maxima.
GRID = [(1, 1, 1), (1, 3, 2), (2, 5, 1), (7, 7, 7), (31, 1, 1), (64, 1, 4), (63, 3, 2), (96, 3, 2), (129, 2, 5),
        (17, 4, 1), (255, 1, 8), (40, 5, 3), (127, 1, 1), (30, 4, 6), (48, 6, 4), (4096, 1, 1), (4096, 256, 1),
        (300, 1, 256), (513, 256, 255)]


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def taps(ntaps, up, down):
    if ntaps == 1:
        return np.array([0.7])
    return signal.firwin(ntaps, 0.8 / max(up, down))


def hard_input(rng, nstreams, n):
    """Gaussian frames with runs of +0, -0, (-0, +0), subnormals and large values."""
    x = (rng.standard_normal((nstreams, n)) + 1j * rng.standard_normal((nstreams, n))).astype(np.complex64)
    m = n // 8
    x[:, m:2 * m] = 0
    x[:, 2 * m:2 * m + m // 4] = np.complex64(complex(-0.0, -0.0))
    x[:, 3 * m:3 * m + m // 4] = np.complex64(complex(-0.0, 0.0))
    sub = rng.integers(1, 1 << 23, size=(nstreams, m // 2)).astype(np.uint32).view(np.float32)
    x.real[:, 4 * m:4 * m + m // 2] = sub
    x.imag[:, 4 * m:4 * m + m // 2] = -sub
    x[:, 5 * m:5 * m + m // 2] *= np.float32(3e37)
    return x


def feed_in_pieces(st, x, rng, longest):
    outs, i = [], 0
    while i < x.shape[1]:
        k = int(rng.integers(1, longest + 1))
        outs.append(st.feed(x[:, i:i + k]))
        i += k
    return np.concatenate(outs, axis=1)


@pytest.mark.parametrize("ntaps,up,down", GRID)
def test_streaming_restatement_is_upfirdn(ntaps, up, down):
    rng = np.random.default_rng(ntaps * 1000 + up * 10 + down)
    h = taps(ntaps, up, down)
    hp = -(-ntaps // up)
    n = 3000 if ntaps < 1000 else 1200
    x = hard_input(rng, 2, n)
    st = sxfir.Stream(h, up, down, nstreams=2)
    # pieces shorter than the history, single frames, and long ones
    y = feed_in_pieces(st, x, rng, max(2, min(300, 2 * hp)))
    assert y.shape[1] == -(-n * up // down)
    # upfirdn's flush tail is what feeding zeros gives.  With few taps, ceil(n up / down) can exceed
    # upfirdn's own length: those outputs are upfirdn of the input followed by zeros.
    tail = st.feed(np.zeros((2, hp + down), np.complex64))
    full = np.concatenate([y, tail], axis=1)
    for s in range(2):
        want = signal.upfirdn(h.astype(np.float32), x[s], up, down)
        padded = signal.upfirdn(h.astype(np.float32), np.concatenate([x[s], np.zeros(2 * (hp + down), np.complex64)]), up, down)
        assert want.dtype == np.complex64
        assert same_bits(y[s], padded[:y.shape[1]]), s
        assert same_bits(full[s], padded[:full.shape[1]]), s
        assert same_bits(full[s, :want.size], want), s


@pytest.mark.parametrize("ntaps,up,down", [(64, 1, 4), (63, 3, 2), (40, 5, 3), (7, 7, 7)])
def test_output_counts_and_phase(ntaps, up, down):
    rng = np.random.default_rng(5)
    st = sxfir.Stream(taps(ntaps, up, down), up, down)
    fed = emitted = 0
    for _ in range(200):
        k = int(rng.integers(1, 40))
        want = sxfir.output_frames(fed, k, up, down)
        assert want == sxfir.output_frames(fed % down, k, up, down)  # the phase alone decides
        y = st.feed(np.zeros((1, k), np.complex64))
        assert y.shape[1] == want
        fed += k
        emitted += want
        assert emitted == -(-fed * up // down) and st.phase == fed % down


def test_state_restores_on_a_second_stream_object():
    rng = np.random.default_rng(6)
    h = taps(63, 3, 2)
    x = hard_input(rng, 3, 900)
    a = sxfir.Stream(h, 3, 2, nstreams=3)
    a.feed(x[:, :401])
    b = sxfir.Stream(h, 3, 2, nstreams=3)
    b.set_state(a.hist, a.phase)
    assert same_bits(a.feed(x[:, 401:]), b.feed(x[:, 401:]))


def fir_kernels_sass():
    """{kernel name: SASS text} of the kernels of libsxgpu.so whose names contain "fir"."""
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
    return {k: "\n".join(v) for k, v in kernels.items() if "fir" in k}


def test_fir_kernels_have_no_fused_multiply_add():
    kernels = fir_kernels_sass()
    assert any("fir_apply_kernel" in k for k in kernels), sorted(kernels)
    for name, sass in kernels.items():
        assert not re.search(r"\bFFMA2?\b", sass), name
        if "fir_apply_kernel" in name:
            assert re.search(r"\bFMUL2?\b", sass) and re.search(r"\bFADD2?\b", sass), name

"""CPU: the numpy restatement of sxgpu_nco_* (tests/sxnco.py), which the GPU tests compare the kernels
against bit for bit, is the oscillator it claims to be: its phasor is within 3.5e-6 of
exp(2 pi j phi / 2^32) at every 20-bit phase step and its worst offsets, its tables cannot depend on
which accurate libm built them, frequencies quantise as the header says, and a sequence fed in any
split into calls equals one call.  And the oscillator kernels in libsxgpu.so contain no fused
multiply-add, which would change the bits."""
import math
import re

import numpy as np
import pytest

import sxnco
from test_fir_oracle import same_bits

PHASOR_ERROR = 3.5e-6


def exact(phi):
    return np.exp(2j * np.pi * np.asarray(phi, np.float64) / 2**32)


def as_complex(cs):
    c, s = cs
    assert c.dtype == np.float32 and s.dtype == np.float32
    return c.astype(np.float64) + 1j * s.astype(np.float64)


def test_phasor_error_at_every_step_and_its_worst_offsets():
    u = np.arange(2**20, dtype=np.int64)
    worst = 0.0
    for off in (-2048, -2047, 0, 2047):
        phi = ((u << 12) + off) % 2**32
        worst = max(worst, float(np.abs(as_complex(sxnco.phasor(phi.astype(np.uint32))) - exact(phi)).max()))
    phi = np.random.default_rng(1).integers(0, 2**32, 1 << 22, dtype=np.uint64).astype(np.uint32)
    worst = max(worst, float(np.abs(as_complex(sxnco.phasor(phi)) - exact(phi)).max()))
    assert worst < PHASOR_ERROR, worst
    assert worst > 1e-7, worst  # the phase is rounded to 20 bits: a phasor this close would be suspicious


def test_rounding_to_twenty_bits_is_to_nearest():
    """Phases within 2048 below and 2047 above a step u 2^12 give the phasor of that step."""
    for u in (0, 1, 1023, 1024, 2**19, 2**20 - 1):
        base = (u << 12) % 2**32
        phi = np.array([(base - 2048) % 2**32, base, (base + 2047) % 2**32], np.uint64).astype(np.uint32)
        c, s = sxnco.phasor(phi)
        assert len(set(c.view(np.uint32).tolist())) == 1 and len(set(s.view(np.uint32).tolist())) == 1, u
    c, s = sxnco.phasor(np.array([0, 2**32 - 2048], np.uint64).astype(np.uint32))  # wraps to step 0
    assert c[0] == c[1] == 1.0 and s[0] == s[1] == 0.0


def test_tables_are_far_from_float32_rounding_midpoints():
    """No entry's double value lies within 2^-50 (relative) of a point half-way between two float32
    values, so any libm accurate to 1 ulp rounds it to the same float32."""
    closest = 1.0
    for table in (sxnco.A_DOUBLE, sxnco.B_DOUBLE):
        for x in np.concatenate(table):
            x = float(x)
            f = np.float32(x)
            if x == 0.0 or float(f) == x:
                continue
            other = np.nextafter(f, np.float32(np.inf) if x > float(f) else np.float32(-np.inf))
            closest = min(closest, abs(x - (float(f) + float(other)) / 2) / abs(x))
    assert closest > 2.0**-50, closest


def test_tables_are_the_float32_roundings_of_libm():
    for k in (0, 1, 256, 511, 1023):
        assert sxnco.A_RE[k] == np.float32(math.cos(2.0 * math.pi * k / 1024.0))
        assert sxnco.B_IM[k] == np.float32(math.sin(2.0 * math.pi * k / 1048576.0))
    assert sxnco.A_RE[0] == 1.0 and sxnco.A_IM[256] == 1.0 and sxnco.A_RE[512] == -1.0


def test_frequency_quantisation():
    q = lambda f: int(sxnco.increments([f], 1)[0])  # noqa: E731
    assert q(0.0) == 0 and q(-0.0) == 0
    assert q(0.5) == 2**31 and q(-0.5) == 2**31
    assert q(0.25) == 2**30 and q(-0.25) == 3 * 2**30
    assert q(1.0 / 2**32) == 1 and q(-1.0 / 2**32) == 2**32 - 1
    # exactly half-way between two increments: to the even one
    assert q(0.5 / 2**32) == 0 and q(1.5 / 2**32) == 2 and q(2.5 / 2**32) == 2 and q(3.5 / 2**32) == 4
    assert q(-0.5 / 2**32) == 0 and q(-1.5 / 2**32) == 2**32 - 2
    assert q(0.1) == round(0.1 * 2**32)
    for bad in (0.5000001, -0.51, math.inf, -math.inf, math.nan):
        with pytest.raises(ValueError):
            sxnco.increments([bad], 1)


def test_mixing_moves_a_tone():
    """A tone at +f0 tuned by -f0 comes out at DC: the sign convention of the header."""
    f0 = 0.1234
    n = np.arange(4096)
    x = (0.5 * np.exp(2j * np.pi * f0 * n)).astype(np.complex64)
    y = sxnco.Stream(1, [-f0]).feed(x[None])[0]
    assert np.abs(y - 0.5).max() < 1e-4
    assert np.abs(np.abs(y) - 0.5).max() < 1e-5


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_any_split_equals_one_call(seed):
    rng = np.random.default_rng(seed)
    S, n = 3, 5000
    freqs = rng.uniform(-0.5, 0.5, S)
    x = (rng.standard_normal((S, n)) + 1j * rng.standard_normal((S, n))).astype(np.complex64)
    whole = sxnco.Stream(S, freqs)
    want = whole.feed(x)
    parts, i, st = [], 0, sxnco.Stream(S, freqs)
    while i < n:
        k = int(rng.integers(1, 400))
        parts.append(st.feed(x[:, i:i + k]))
        i += k
    assert same_bits(np.concatenate(parts, axis=1), want)
    assert np.array_equal(st.phase, whole.phase) and np.array_equal(st.inc, whole.inc)


def test_phase_wraps_over_two_to_the_32_frames():
    """A call of 2^32 + m frames: frame k of it sees the phase that a call starting k frames later
    starts with, and the phase after it is that of a call of m frames.  (Frames past 2^32 are
    checked through the phase formula; 2^32 frames do not fit here.)"""
    inc = sxnco.increments([0.3, -0.123456789, 0.5], 3)
    start = np.array([2**32 - 5, 17, 2**31], np.uint32)
    k = np.array([0, 1, 2**31, 2**32 - 1, 2**32, 2**32 + 1, 2**32 + 77, 3 * 2**32 + 5], np.uint64)
    ph = sxnco.phases(start, inc, k)
    for j, kk in enumerate(k.tolist()):
        st = sxnco.Stream(3)
        st.phase, st.inc = start.copy(), inc.copy()
        st.skip(kk)
        assert np.array_equal(st.phase, ph[:, j]), kk
    assert np.array_equal(ph[:, 4], start)
    assert np.array_equal(ph[:, 6], sxnco.phases(start, inc, [77])[:, 0])
    assert np.array_equal(ph[:, 7], sxnco.phases(start, inc, [5])[:, 0])
    # fed in pieces across a 32-bit phase wrap
    x = np.ones((3, 64), np.complex64)
    a, b = sxnco.Stream(3), sxnco.Stream(3)
    for st in (a, b):
        st.phase, st.inc = start.copy(), inc.copy()
    assert same_bits(a.feed(x), np.concatenate([b.feed(x[:, :7]), b.feed(x[:, 7:])], axis=1))


def test_retune_keeps_the_phase_continuous():
    st = sxnco.Stream(1, [0.01])
    st.feed(np.ones((1, 100), np.complex64))
    before = int(st.phase[0])
    assert before == 100 * int(sxnco.increments([0.01], 1)[0]) % 2**32
    st.retune([-0.2])
    y = st.feed(np.ones((1, 1), np.complex64))
    assert same_bits(y, sxnco.mix(np.ones((1, 1), np.complex64), np.array([[before]], np.uint32)))


def nco_kernels_sass():
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
    # the mixing instantiations of the FIR kernels have NcoView among their template arguments
    return {k: "\n".join(v) for k, v in kernels.items() if "nco" in k or "NcoView" in k}


def test_nco_and_mixing_fir_kernels_have_no_fused_multiply_add():
    kernels = nco_kernels_sass()
    assert any("nco_apply_kernel" in k for k in kernels), sorted(kernels)
    assert any("nco_advance_kernel" in k for k in kernels), sorted(kernels)
    for must in ("bank_fir_kernel", "bank_fir_read_tail_kernel", "fir_history_kernel"):
        assert any(must in k and "NcoView" in k for k in kernels), (must, sorted(kernels))
    assert sum("bank_fir_kernel" in k for k in kernels) == 6, sorted(kernels)  # R = 1, 2, 4, read and write
    for name, sass in kernels.items():
        assert not re.search(r"\bFFMA2?\b", sass), name
        if "apply" in name or "bank_fir_kernel" in name or "read_tail" in name:
            assert re.search(r"\bFMUL2?\b", sass) and re.search(r"\bFADD2?\b", sass), name

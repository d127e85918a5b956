"""numpy restatement of sxgpu_nco_* (include/sxgpu.h, sxxcvr_b200/csrc/sx_nco.cuh), the specification
the GPU tests compare against bit for bit.

Per stream a 32-bit phase phi_s and a 32-bit increment inc_s.  Frame k of a call is multiplied by
the phasor of phi = phi_s + (k mod 2^32) inc_s (mod 2^32); a call of n frames then adds n inc_s to
phi_s.  A frequency f (cycles per sample) becomes inc = rint(f 2^32) mod 2^32, half to even.

The phasor is a two-table lookup rounded to 20 bits of phase:
    u = ((phi + 2048) mod 2^32) >> 12,  hi = u >> 10,  lo = u & 1023
    A[hi] = e^{j 2 pi hi / 1024},  B[lo] = e^{j 2 pi lo / 2^20}    (libm double cos / sin, rounded once)
    c = A.re B.re - A.im B.im,  s = A.im B.re + A.re B.im
    y.re = x.re c - x.im s,     y.im = x.re s + x.im c
every product and sum one float32 rounding.  ddc() and duc() compose it with tests/sxfir.py as
sxgpu_bank_read_ddc and sxgpu_bank_write_duc do.
"""
from __future__ import annotations

import math

import numpy as np

TABLE = 1024


def _table(denominator):
    re = np.array([math.cos(2.0 * math.pi * k / denominator) for k in range(TABLE)], np.float64)
    im = np.array([math.sin(2.0 * math.pi * k / denominator) for k in range(TABLE)], np.float64)
    return re, im


A_DOUBLE = _table(1024.0)
B_DOUBLE = _table(1048576.0)
A_RE, A_IM = (t.astype(np.float32) for t in A_DOUBLE)
B_RE, B_IM = (t.astype(np.float32) for t in B_DOUBLE)


def increments(freqs, nstreams):
    """rint(f 2^32) mod 2^32 per stream, as uint32; refuses what sxgpu_nco_create refuses."""
    f = np.broadcast_to(np.asarray(freqs, np.float64), (nstreams,))
    if not np.isfinite(f).all() or (np.abs(f) > 0.5).any():
        raise ValueError("frequencies are finite and within -0.5 .. 0.5")
    return (np.rint(f * 2.0**32).astype(np.int64) % 2**32).astype(np.uint32)


def phasor(phi):
    """(c, s) float32 of uint32 phases."""
    u = (np.asarray(phi, np.uint32).astype(np.uint64) + 2048) % 2**32 >> 12
    hi, lo = (u >> 10).astype(np.intp), (u & 1023).astype(np.intp)
    ar, ai, br, bi = A_RE[hi], A_IM[hi], B_RE[lo], B_IM[lo]
    return ar * br - ai * bi, ai * br + ar * bi


def mix(x, phi):
    """x (complex64) times the phasor of phi, elementwise."""
    x = np.asarray(x, np.complex64)
    c, s = phasor(phi)
    xr, xi = x.real, x.imag
    y = np.empty(x.shape, np.complex64)
    y.real = xr * c - xi * s
    y.imag = xr * s + xi * c
    return y


def phases(phase, inc, k):
    """The phase of frame(s) k of a call that starts at `phase`: phase + (k mod 2^32) inc mod 2^32."""
    k = np.asarray(k, np.uint64) % 2**32
    return ((np.asarray(phase, np.uint64)[..., None] + k * np.asarray(inc, np.uint64)[..., None]) % 2**32).astype(np.uint32)


class Stream:
    """The oscillators of `nstreams` streams: one phase and one increment each."""

    def __init__(self, nstreams=1, freqs=None):
        self.nstreams = nstreams
        self.phase = np.zeros(nstreams, np.uint32)
        self.inc = increments(0.0 if freqs is None else freqs, nstreams)

    def retune(self, freqs):
        """As sxgpu_nco_set_frequencies: new increments, the phases kept."""
        self.inc = increments(0.0 if freqs is None else freqs, self.nstreams)

    def skip(self, n):
        """The phases after a call of n frames, without the frames."""
        self.phase = ((self.phase.astype(np.uint64) + (n % 2**32) * self.inc.astype(np.uint64)) % 2**32).astype(np.uint32)

    def feed(self, x):
        """x: (nstreams, n) complex64 -> the same frames mixed; the phases advance by n inc."""
        x = np.asarray(x, np.complex64).reshape(self.nstreams, -1)
        y = mix(x, phases(self.phase, self.inc, np.arange(x.shape[1], dtype=np.uint64)))
        self.skip(x.shape[1])
        return y


def ddc(nco, fir, x):
    """sxgpu_bank_read_ddc on the block the bank read: mix, then filter (fir: a tests/sxfir.py Stream)."""
    return fir.feed(nco.feed(x))


def duc(fir, nco, x):
    """sxgpu_bank_write_duc before the bank's conversion: filter, then mix."""
    return nco.feed(fir.feed(x))

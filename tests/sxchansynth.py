"""numpy restatement of sxgpu_chan_synth_* (include/sxgpu.h, sxxcvr_b200/csrc/sx_chan.cuh), the
specification the GPU tests compare against bit for bit.

M channels (a power of two), interpolation D dividing M, real taps h rounded to float32 once, hp =
ceil(ntaps / D).  X counts the input frames per channel fed; frames before the first are 0.  For
output frame n = m D + t (t < D) of a stream:
    1. Y_m = the unnormalised inverse DFT of (y_0[m] .. y_{M-1}[m]): a[i] = y_{rev(i)}[m], rev
       reversing the log2 M bits of i; radix-2 decimation in time, h = 1, 2, .. M/2, for every i
       with (i mod 2h) < h:
           w = T+[(i mod 2h) M / (2h)],  p = a[i],  q = a[i+h]
           t.re = q.re w.re - q.im w.im,  t.im = q.re w.im + q.im w.re
           a[i] = p + t,  a[i+h] = p - t
       T+[j] = A[j 1024 / M], the oscillator's coarse table (tests/sxnco.py), not conjugated;
       Y_m[i] = a[i]
    2. acc = +0;  for p = P_t - 1 down to 0:  acc = acc + Y_{m-p}[n mod M] * h[t + p D]
       (P_t = ceil((ntaps - t) / D), 0 when t >= ntaps)
every product and sum one float32 rounding, I and Q separately.  Vectorised over streams, frames,
outputs and each stage's butterflies, with loops over the stages and the taps of a phase.
"""
from __future__ import annotations

import numpy as np

import sxnco
from sxchan import bit_reverse


def twiddles(m):
    """(re, im) float32 of T+[j], j < m / 2."""
    q = np.arange(m // 2) * (sxnco.TABLE // m)
    return sxnco.A_RE[q], sxnco.A_IM[q]


def idft(yr, yi, m):
    """Step 1 on channel values (..., m) float32: (Y.re, Y.im), (..., m)."""
    bits = m.bit_length() - 1
    rev = bit_reverse(np.arange(m), bits)
    ar, ai = np.array(yr[..., rev], np.float32), np.array(yi[..., rev], np.float32)
    tr_, ti_ = twiddles(m)
    h = 1
    while h < m:
        # i = 2h g + jj, jj < h: p = a[i], q = a[i + h], w = T+[jj M / (2h)]
        vr, vi = ar.reshape(*ar.shape[:-1], m // (2 * h), 2, h), ai.reshape(*ai.shape[:-1], m // (2 * h), 2, h)
        w = np.arange(h) * (m // (2 * h))
        wr, wi = tr_[w], ti_[w]
        pr, pi, qr, qi = vr[..., 0, :], vi[..., 0, :], vr[..., 1, :], vi[..., 1, :]
        tr = qr * wr - qi * wi
        ti = qr * wi + qi * wr
        qr[...], qi[...] = pr - tr, pi - ti
        pr += tr
        pi += ti
        h *= 2
    return ar, ai


class Stream:
    """The synthesizer state of `nstreams` streams: each channel's last hp - 1 inputs (oldest first)
    and the input frames fed so far."""

    def __init__(self, h, channels, up=None, nstreams=1):
        self.h = np.asarray(h, np.float64).astype(np.float32)
        self.m, self.up, self.nstreams = channels, channels if up is None else up, nstreams
        self.ntaps = self.h.size
        self.hp = -(-self.ntaps // self.up)
        self.hist = np.zeros((nstreams, channels, self.hp - 1), np.complex64)
        self.fed = 0

    @property
    def phase(self):
        return self.fed % (self.m // self.up)

    def set_state(self, hist=None, phase=0):
        """As sxgpu_chan_synth_set_state: only the frame count mod M / D matters from here on."""
        shape = (self.nstreams, self.m, self.hp - 1)
        self.hist = np.zeros(shape, np.complex64) if hist is None else np.array(hist, np.complex64).reshape(shape)
        self.fed = phase

    def feed(self, y):
        """y: (nstreams, M, nin) complex64 -> (nstreams, nin D) complex64, the history carried."""
        m, d, hp = self.m, self.up, self.hp
        y = np.asarray(y, np.complex64).reshape(self.nstreams, m, -1)
        nin = y.shape[2]
        buf = np.concatenate([self.hist, y], axis=2)  # column b holds channel frame fed - (hp - 1) + b
        frames = np.ascontiguousarray(buf.transpose(0, 2, 1))  # (streams, buffer frames, M)
        yr, yi = idft(frames.real, frames.imag, m)
        # output o = j D + t reads column n mod M = q D + t, q = (phase + j) mod P (P = M / D), of
        # buffer frame b = j + hp - 1 - p, so q = (phase + b - hp + 1 + p) mod P: with the blocks
        # gathered once per shift r = p mod P, every tap p reads a contiguous run of frames.
        P, nbuf = m // d, nin + hp - 1
        b = np.arange(nbuf)
        q = (self.phase + b[None, :] - hp + 1 + np.arange(P)[:, None]) % P  # (r, b)
        gr = yr.reshape(self.nstreams, nbuf, P, d)[:, b[None, :], q, :]  # (streams, r, b, t)
        gi = yi.reshape(self.nstreams, nbuf, P, d)[:, b[None, :], q, :]
        t = np.arange(d)
        ntap = np.where(t < self.ntaps, -(-(self.ntaps - t) // d), 0)
        ar = np.zeros((self.nstreams, nin, d), np.float32)
        ai = np.zeros((self.nstreams, nin, d), np.float32)
        hpad = np.zeros(hp * d, np.float32)
        hpad[:self.ntaps] = self.h
        for p in range(hp - 1, -1, -1):
            live = p < ntap  # only the taps that exist are multiplied
            hv = hpad[t + p * d]
            for acc, part in ((ar, gr), (ai, gi)):
                prod = part[:, p % P, hp - 1 - p:hp - 1 - p + nin, :] * hv
                if live.all():
                    acc += prod
                else:
                    acc[..., live] += prod[..., live]
        self.fed += nin
        if hp > 1:
            self.hist = np.ascontiguousarray(buf[:, :, buf.shape[2] - (hp - 1):])
        x = np.empty((self.nstreams, nin * d), np.complex64)
        x.real, x.imag = ar.reshape(self.nstreams, -1), ai.reshape(self.nstreams, -1)
        return x


def definition(h, y, channels, up):
    """The float64 definition for channels fed y from frame 0: (nstreams, nin D) complex128,
    x[n] = sum_k sum_m h[n - m D] y_k[m] e^{+j 2 pi k n / M}."""
    h = np.asarray(h, np.float64).astype(np.float32).astype(np.float64)
    y = np.asarray(y, np.complex128)
    nstreams, m, nin = y.shape
    n = np.arange(nin * up)
    x = np.zeros((nstreams, n.size), np.complex128)
    for k in range(m):
        for s in range(nstreams):
            z = np.zeros(n.size, np.complex128)
            z[::up] = y[s, k]
            x[s] += np.convolve(z, h)[:n.size] * np.exp(2j * np.pi * k * (n % m) / m)
    return x

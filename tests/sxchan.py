"""numpy restatement of sxgpu_chan_* (include/sxgpu.h, sxxcvr_b200/csrc/sx_chan.cuh), the
specification the GPU tests compare against bit for bit.

M channels (a power of two), decimation D dividing M, real taps h rounded to float32 once.  X counts
the frames a stream has been fed; frames before the first are 0.  Output m of channel k, N = m D:
    1. u_r = +0;  for p = P_r - 1 down to 0:  u_r = u_r + x[N - p M - r] * h[p M + r]
       (r < M, P_r = ceil((ntaps - r) / M), 0 when r >= ntaps)
    2. a[i] = u_{(N - rev(i)) mod M}, rev reversing the log2 M bits of i
    3. radix-2 decimation in time, h = 1, 2, .. M/2, for every i with (i mod 2h) < h:
           w = T[(i mod 2h) M / (2h)],  p = a[i],  q = a[i+h]
           t.re = q.re w.re - q.im w.im,  t.im = q.re w.im + q.im w.re
           a[i] = p + t,  a[i+h] = p - t
       T[j] = (A.re, -A.im) of the oscillator's coarse table entry A[j 1024 / M] (tests/sxnco.py)
    4. y_k[m] = a[k]
every product and sum one float32 rounding, I and Q separately.  Vectorised over streams, outputs,
branches and each stage's butterflies, with loops over the taps of a branch and over the stages.
"""
from __future__ import annotations

import numpy as np

import sxnco


def twiddles(m):
    """(re, im) float32 of T[j], j < m / 2."""
    q = np.arange(m // 2) * (sxnco.TABLE // m)
    return sxnco.A_RE[q], -sxnco.A_IM[q]


def bit_reverse(i, bits):
    i = np.asarray(i, np.int64)
    out = np.zeros_like(i)
    for b in range(bits):
        out |= ((i >> b) & 1) << (bits - 1 - b)
    return out


def output_frames(fed, nin, down):
    """ceil((fed + nin) / down) - ceil(fed / down)."""
    return -(-(fed + nin) // down) - -(-fed // down)


def dft(ur, ui, nmod, m):
    """Steps 2-4 on branch sums u (..., outputs, m) float32, nmod = N mod m per output: a (..., outputs, m)."""
    bits = m.bit_length() - 1
    src = (nmod[:, None] - bit_reverse(np.arange(m), bits)[None, :]) % m  # (outputs, m)
    ar = np.take_along_axis(ur, np.broadcast_to(src, ur.shape), axis=-1)
    ai = np.take_along_axis(ui, np.broadcast_to(src, ui.shape), axis=-1)
    tr_, ti_ = twiddles(m)
    h = 1
    while h < m:
        i = np.arange(m)
        i = i[(i % (2 * h)) < h]
        j = i + h
        w = (i % (2 * h)) * (m // (2 * h))
        wr, wi = tr_[w], ti_[w]
        pr, pi, qr, qi = ar[..., i], ai[..., i], ar[..., j], ai[..., j]
        tr = qr * wr - qi * wi
        ti = qr * wi + qi * wr
        ar[..., i], ai[..., i] = pr + tr, pi + ti
        ar[..., j], ai[..., j] = pr - tr, pi - ti
        h *= 2
    return ar, ai


class Stream:
    """The channelizer state of `nstreams` streams: the last ntaps - 1 inputs of each (oldest first)
    and the frames fed so far."""

    def __init__(self, h, channels, down=None, nstreams=1):
        self.h = np.asarray(h, np.float64).astype(np.float32)
        self.m, self.down, self.nstreams = channels, channels if down is None else down, nstreams
        self.ntaps = self.h.size
        self.hist = np.zeros((nstreams, self.ntaps - 1), np.complex64)
        self.fed = 0

    @property
    def phase(self):
        return self.fed % self.m

    def set_state(self, hist=None, phase=0):
        """As sxgpu_chan_set_state: only the frame count mod M matters from here on."""
        self.hist = np.zeros((self.nstreams, self.ntaps - 1), np.complex64) if hist is None else \
            np.array(hist, np.complex64).reshape(self.nstreams, self.ntaps - 1)
        self.fed = phase

    def feed(self, x):
        """x: (nstreams, nin) complex64 -> (nstreams, M, nout) complex64, the history carried."""
        x = np.asarray(x, np.complex64).reshape(self.nstreams, -1)
        m, d, ntaps = self.m, self.down, self.ntaps
        buf = np.concatenate([self.hist, x], axis=1)
        # buffer column b holds stream frame self.fed - (ntaps - 1) + b
        first = -(-self.fed // d)
        end = -(-(self.fed + x.shape[1]) // d)
        n = np.arange(first, end, dtype=np.int64) * d
        col = n - self.fed + ntaps - 1
        re, im = np.ascontiguousarray(buf.real), np.ascontiguousarray(buf.imag)
        ur = np.zeros((self.nstreams, n.size, m), np.float32)
        ui = np.zeros((self.nstreams, n.size, m), np.float32)
        for p in range(-(-ntaps // m) - 1, -1, -1) if n.size else ():
            live = min(m, ntaps - p * m)  # the branches r < live have a tap p
            hv = self.h[p * m:p * m + live]
            for acc, part in ((ur, re), (ui, im)):
                # frames col[o] - p m - r: a view with stride D along o and -1 along r
                start = part[:, col[0] - p * m:]
                s0, s1 = part.strides
                xv = np.lib.stride_tricks.as_strided(start, (self.nstreams, n.size, live), (s0, d * s1, -s1))
                acc[:, :, :live] += xv * hv
        ar, ai = dft(ur, ui, n % m, m)
        self.fed += x.shape[1]
        if ntaps > 1:
            self.hist = np.ascontiguousarray(buf[:, buf.shape[1] - (ntaps - 1):])
        y = np.empty((self.nstreams, m, n.size), np.complex64)
        y.real, y.imag = ar.transpose(0, 2, 1), ai.transpose(0, 2, 1)
        return y


def definition(h, x, channels, down):
    """The float64 definition for a stream fed x from frame 0: (nstreams, M, ceil(nin / D)) complex128."""
    h = np.asarray(h, np.float64).astype(np.float32).astype(np.float64)
    x = np.asarray(x, np.complex128).reshape(-1, np.shape(x)[-1])
    nin, ntaps = x.shape[1], h.size
    n = np.arange(0, nin, down)
    j = np.arange(ntaps)
    idx = n[:, None] - j[None, :]
    xx = np.where(idx >= 0, x[:, np.clip(idx, 0, None)], 0)  # (streams, outputs, taps)
    k = np.arange(channels)
    ph = np.exp(-2j * np.pi * np.outer(k, idx.reshape(-1) % channels) / channels).reshape(channels, *idx.shape)
    return np.einsum("sot,t,kot->sko", xx, h, ph)

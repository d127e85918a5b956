"""numpy restatement of sxgpu_fir_apply (include/sxgpu.h, sxxcvr_b200/csrc/sx_fir.cuh), the
specification the GPU tests compare against bit for bit.

A stream fed X frames in total has emitted the first ceil(X up / down) outputs of
scipy.signal.upfirdn(h.astype(float32), x.astype(complex64), up, down).  Polyphase, hp =
ceil(ntaps / up) taps per phase, h zero-padded to hp up; output n reads the inputs ending at
newest = (n down) // up with the taps of phase t = (n down) % up, oldest first, each product and
each sum one float32 rounding:

    acc = +0;  for j = hp-1 down to 0:  acc = acc + x[newest - j] * h[t + up j]    (x before 0 is 0)

I and Q are filtered independently by the same real taps.  Vectorised over streams and outputs,
with a loop over the taps.
"""
from __future__ import annotations

import numpy as np


def polyphase(h, up):
    """h rounded to float32 and zero-padded to hp * up taps."""
    h = np.asarray(h, np.float64).astype(np.float32)
    hp = -(-h.size // up)
    hpad = np.zeros(hp * up, np.float32)
    hpad[:h.size] = h
    return hpad, hp


def output_frames(fed, nin, up, down):
    """Outputs a call of nin frames emits after `fed` frames: ceil((fed + nin) up / down) - ceil(fed up / down)."""
    return -(-(fed + nin) * up // down) - -(-fed * up // down)


class Stream:
    """The FIR state of `nstreams` streams: the last hp - 1 inputs of each (oldest first) and the
    frames fed so far."""

    def __init__(self, h, up=1, down=1, nstreams=1):
        self.hpad, self.hp = polyphase(h, up)
        self.up, self.down, self.nstreams = up, down, nstreams
        self.hist = np.zeros((nstreams, self.hp - 1), np.complex64)
        self.fed = 0

    @property
    def phase(self):
        return self.fed % self.down

    def set_state(self, hist=None, phase=0):
        """As sxgpu_fir_set_state: only the phase of the frame count matters from here on."""
        self.hist = np.zeros((self.nstreams, self.hp - 1), np.complex64) if hist is None else \
            np.array(hist, np.complex64).reshape(self.nstreams, self.hp - 1)
        self.fed = phase

    def feed(self, x):
        """x: (nstreams, nin) complex64 -> (nstreams, nout) complex64, the history carried."""
        x = np.asarray(x, np.complex64).reshape(self.nstreams, -1)
        up, down, hp = self.up, self.down, self.hp
        buf = np.concatenate([self.hist, x], axis=1)
        # buffer column b holds stream frame self.fed - (hp - 1) + b
        first = -(-self.fed * up // down)
        end = -(-(self.fed + x.shape[1]) * up // down)
        n = np.arange(first, end, dtype=np.int64)
        t = (n * down) % up
        col = (n * down) // up - self.fed + hp - 1
        re, im = np.ascontiguousarray(buf.real), np.ascontiguousarray(buf.imag)
        ar = np.zeros((self.nstreams, n.size), np.float32)
        ai = np.zeros((self.nstreams, n.size), np.float32)
        for j in range(hp - 1, -1, -1):
            hv = self.hpad[t + up * j]
            ar = ar + re[:, col - j] * hv
            ai = ai + im[:, col - j] * hv
        self.fed += x.shape[1]
        if hp > 1:
            self.hist = np.ascontiguousarray(buf[:, buf.shape[1] - (hp - 1):])
        y = np.empty((self.nstreams, n.size), np.complex64)
        y.real, y.imag = ar, ai
        return y

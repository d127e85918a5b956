"""A numpy restatement of the bank's IIR filters (sxxcvr_b200/csrc/sx_iir.cuh): cascaded
second-order sections in scipy's transposed direct form II, float32, applied to the real and
the imaginary part of complex64 samples independently with the same real coefficients.

For one sample x of one component and one section (b0 b1 b2 1 a1 a2), in this order, every
operation a single correctly rounded float32 operation:

    y  = b0*x + z0
    z0 = (b1*x - a1*y) + z1
    z1 = b2*x - a2*y

numpy evaluates float32 arrays exactly so (it never contracts a multiply and an add), and the
loop runs over frames with every stream and component of a frame at once."""
from __future__ import annotations

import numpy as np

MAX_SECTIONS = 8


def sos32(sos) -> np.ndarray:
    """Coefficients as the library holds them: float64 input rounded to float32 once."""
    return np.asarray(sos, dtype=np.float64).reshape(-1, 6).astype(np.float32)


def sosfilt(sos, x: np.ndarray, zi: np.ndarray | None = None):
    """sosfilt(sos, x, zi) along the last axis of complex64 x of shape (nstreams, n).

    zi, and the returned zf: (nsections, nstreams, 2) complex64, scipy's layout.  Returns (y, zf)."""
    c = sos32(sos)
    x = np.ascontiguousarray(x, dtype=np.complex64)
    nstreams, n = x.shape
    xf = x.view(np.float32).reshape(nstreams, n, 2)
    z = np.zeros((c.shape[0], nstreams, 2, 2), np.float32) if zi is None else \
        np.ascontiguousarray(zi, dtype=np.complex64).view(np.float32).reshape(c.shape[0], nstreams, 2, 2).copy()
    y = np.empty_like(xf)
    for t in range(n):
        cur = xf[:, t, :]
        for k in range(c.shape[0]):
            b0, b1, b2, _, a1, a2 = c[k]
            out = b0 * cur + z[k, :, 0, :]
            z[k, :, 0, :] = (b1 * cur - a1 * out) + z[k, :, 1, :]
            z[k, :, 1, :] = b2 * cur - a2 * out
            cur = out
        y[:, t, :] = cur
    return y.reshape(nstreams, n * 2).view(np.complex64), z.reshape(c.shape[0], nstreams, 4).view(np.complex64)

"""A numpy restatement of sxgpu_iir_apply_long (sxxcvr_b200/csrc/sx_iir.cuh), the specification the
GPU tests hold the library to bit for bit.

Each stream of x[nstreams][nframes] is cut into K = ceil(nframes / L) chunks of L frames (the last
may be shorter).  Pass 1 runs every chunk but a stream's last from a zero state through the float32
cascade of tests/sxiir.py and keeps its end state e_k.  The carry, in float64, per stream and
component: v_0 = zi, v_k = e_{k-1}, s_0 = v_0 and s_k = M s_{k-1} + v_k, with M = A^L and A the
cascade's one-step state matrix (state index 2 q + j for z_j of section q).  Pass 3 runs every
chunk from float32(s_k); a stream's last chunk leaves the filter state.

Evaluation order of the carry: every product and sum is one correctly rounded float64 operation
(numpy's elementwise float64 ufuncs; no BLAS, nothing contracted), a matrix-vector product sums
its columns left to right, a step is (P x) + v, and P_j = A^(2^j) by repeated squaring.  Elements go
in groups of GROUP chunks: a sequential reduce to the group totals, a Hillis-Steele scan over the
totals with P_{log2(L) + 6 + level}, and a sequential fix-up from the previous group's total."""
from __future__ import annotations

import numpy as np

import sxiir

GROUP, LOG2_GROUP = 64, 6
POWERS = 64


def chunk_len(nstreams: int, nframes: int) -> int:
    """L: 1024, halved while nstreams * ceil(nframes / L) < 65536 and L > 128."""
    n = 1024
    while n > 128 and nstreams * (-(-nframes // n)) < 65536:
        n //= 2
    return n


def state_matrix(sos) -> np.ndarray:
    """A, column by column: one float64 step of the cascade on zero input from a unit state."""
    c = sxiir.sos32(sos)
    nsec = c.shape[0]
    n = 2 * nsec
    a = np.zeros((n, n))
    for col in range(n):
        z = [0.0] * n
        z[col] = 1.0
        x = 0.0
        for q in range(nsec):
            b0, b1, b2, _, a1, a2 = (float(v) for v in c[q])
            y = b0 * x + z[2 * q]
            z0 = (b1 * x - a1 * y) + z[2 * q + 1]
            z1 = b2 * x - a2 * y
            z[2 * q], z[2 * q + 1], x = z0, z1, y
        a[:, col] = z
    return a


def matmul(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """x y, each entry summed left to right."""
    acc = x[:, 0:1] * y[0:1, :]
    for m in range(1, x.shape[1]):
        acc = acc + x[:, m:m + 1] * y[m:m + 1, :]
    return acc


def power_chain(sos, count: int = POWERS) -> list[np.ndarray]:
    """P_0 = A, P_{j+1} = P_j P_j."""
    p = [state_matrix(sos)]
    while len(p) < count:
        p.append(matmul(p[-1], p[-1]))
    return p


def matvec(p: np.ndarray, x: np.ndarray) -> np.ndarray:
    """(P x) over the last axis of x, columns summed left to right."""
    acc = x[..., 0:1] * p[:, 0]
    for col in range(1, p.shape[1]):
        acc = acc + x[..., col:col + 1] * p[:, col]
    return acc


def _vectors(z: np.ndarray) -> np.ndarray:
    """scipy's (nsections, rows, 2) complex64 -> (rows, 2 components, 2 nsections) float64."""
    nsec, rows = z.shape[0], z.shape[1]
    f = np.ascontiguousarray(z, dtype=np.complex64).view(np.float32).reshape(nsec, rows, 2, 2)  # [q][row][j][c]
    return f.transpose(1, 3, 0, 2).reshape(rows, 2, 2 * nsec).astype(np.float64)


def _states(v: np.ndarray) -> np.ndarray:
    """The inverse of _vectors, rounding float64 to float32."""
    rows, _, n = v.shape
    f = v.astype(np.float32).reshape(rows, 2, n // 2, 2).transpose(2, 0, 3, 1)  # [q][row][j][c]
    return np.ascontiguousarray(f).view(np.complex64).reshape(n // 2, rows, 2)


def carry(p: list[np.ndarray], v: np.ndarray, log2_len: int) -> np.ndarray:
    """Start states s (nstreams, K, 2, n) from the elements v (same shape), in the kernels' order."""
    nstreams, k, _, n = v.shape
    groups = -(-k // GROUP)
    # The last group is padded with zeros: its total differs from the kernels', and nothing reads it.
    vp = np.concatenate([v, np.zeros((nstreams, groups * GROUP - k, 2, n))], axis=1).reshape(nstreams, groups, GROUP, 2, n)
    m = p[log2_len]
    t = vp[:, :, 0]
    for r in range(1, GROUP):
        t = matvec(m, t) + vp[:, :, r]
    w, level = t, 0
    while (1 << level) < groups:
        d = 1 << level
        nxt = w.copy()
        nxt[:, d:] = matvec(p[log2_len + LOG2_GROUP + level], w[:, :-d]) + w[:, d:]
        w, level = nxt, level + 1
    s = np.empty_like(vp)
    x = vp[:, :, 0].copy()
    x[:, 1:] = matvec(m, w[:, :-1]) + vp[:, 1:, 0]
    s[:, :, 0] = x
    for r in range(1, GROUP):
        x = matvec(m, x) + vp[:, :, r]
        s[:, :, r] = x
    return s.reshape(nstreams, groups * GROUP, 2, n)[:, :k]


def apply_long(sos, x: np.ndarray, zi: np.ndarray | None = None, length: int | None = None, chain=None):
    """sxgpu_iir_apply_long on complex64 x (nstreams, nframes); zi and the returned zf in scipy's
    (nsections, nstreams, 2) complex64 layout.  `length` overrides the chunk rule.  Returns (y, zf)."""
    x = np.ascontiguousarray(x, dtype=np.complex64)
    nstreams, nframes = x.shape
    nsec = sxiir.sos32(sos).shape[0]
    size = chunk_len(nstreams, nframes) if length is None else length
    k = -(-nframes // size)
    if k == 1:
        return sxiir.sosfilt(sos, x, zi)
    if zi is None:
        zi = np.zeros((nsec, nstreams, 2), np.complex64)
    head = (k - 1) * size
    _, ends = sxiir.sosfilt(sos, x[:, :head].reshape(nstreams * (k - 1), size))
    v = np.empty((nstreams, k, 2, 2 * nsec))
    v[:, 0] = _vectors(zi)
    v[:, 1:] = _vectors(ends).reshape(nstreams, k - 1, 2, 2 * nsec)
    s = carry(chain if chain is not None else power_chain(sos), v, size.bit_length() - 1)
    y = np.empty_like(x)
    body, _ = sxiir.sosfilt(sos, x[:, :head].reshape(nstreams * (k - 1), size),
                            _states(s[:, :k - 1].reshape(nstreams * (k - 1), 2, 2 * nsec)))
    y[:, :head] = body.reshape(nstreams, head)
    y[:, head:], zf = sxiir.sosfilt(sos, x[:, head:], _states(s[:, k - 1]))
    return y, zf

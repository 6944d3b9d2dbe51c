"""Blockwise CWT of a long recording, the way the reference's scripts call it (test infrastructure).

The reference's CWT scripts hand a long recording to `cwt` / `ssq_cwt` through dask:
`map_overlap(depth=d, boundary="reflect")` over chunks of C samples (tests/cwt_test.py:117-119,187-193 of the
reference).  Block b covers output columns [bC, min((b+1)C, N)); it is the reference's call on the extended input
e_b[j] = x~[bC - d + j], j < len_b + 2d, trimmed to columns [d, d + len_b).  x~ is the recording mirrored with the edge
sample repeated -- np.pad(mode="symmetric"), which is what dask's `overlap.reflect` does for boundary="reflect" (taken
from dask's source: the boundary slices are x[:d][::-1] and x[-d:][::-1]).
"""
import numpy as np

from oracle import ssq_oracle as O


def n_blocks(N, C):
    return (N + C - 1) // C


def block_len(N, C, b):
    return min((b + 1) * C, N) - b * C


def extended_block(x, C, d, b):
    """e_b along axis 0 of x (the recording, [N] or [N, channels]), by the index rule of the stream's device load."""
    N = x.shape[0]
    q = np.arange(b * C - d, b * C + block_len(N, C, b) + d)
    q = np.where(q < 0, -1 - q, q)
    q = np.where(q >= N, 2 * N - 1 - q, q)
    return x[q]


def blockwise_cwt(x, C, d, scales, **kw):
    """Wx [ns, N] of a 1-D recording: each block through oracle.ssq_oracle.cwt, trimmed, concatenated."""
    parts = []
    for b in range(n_blocks(len(x), C)):
        Wx, _, _ = O.cwt(extended_block(np.asarray(x, dtype=np.float64), C, d, b), scales=scales, **kw)
        parts.append(Wx[:, d:d + block_len(len(x), C, b)])
    return np.concatenate(parts, axis=1)


def blockwise_ssq_cwt(x, C, d, scales, **kw):
    """(Tx [ns, N], [ssq_freqs of each block]) of a 1-D recording through oracle.ssq_oracle.ssq_cwt."""
    parts, freqs = [], []
    for b in range(n_blocks(len(x), C)):
        Tx, sf = O.ssq_cwt(extended_block(np.asarray(x, dtype=np.float64), C, d, b), scales=scales, **kw)
        parts.append(Tx[:, d:d + block_len(len(x), C, b)])
        freqs.append(sf)
    return np.concatenate(parts, axis=1), freqs

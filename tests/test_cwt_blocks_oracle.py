"""CPU: the extended block input of the CWT stream (oracle/cwt_blocks.py) is np.pad(mode="symmetric") sliced, the
boundary rule of the reference's dask map_overlap(boundary="reflect") caller; the blockwise oracle is the reference's
call on those blocks."""
import numpy as np
import pytest

from oracle import cwt_blocks as B
from oracle import ssq_oracle as O


@pytest.mark.parametrize("N,C,d", [(1000, 300, 0), (1000, 300, 300), (1000, 300, 57), (1001, 250, 250),
                                   (250, 1000, 100), (40, 64, 40), (7, 3, 3), (1, 1, 1)])
def test_extended_block_is_symmetric_pad(N, C, d):
    x = np.random.default_rng(N + C + d).standard_normal((N, 3))
    padded = np.pad(x, ((d, d), (0, 0)), mode="symmetric")
    for b in range(B.n_blocks(N, C)):
        e = B.extended_block(x, C, d, b)
        ln = B.block_len(N, C, b)
        assert e.shape == (ln + 2 * d, 3)
        assert np.array_equal(e, padded[b * C:b * C + ln + 2 * d])


def test_blockwise_oracle_is_the_call_on_each_block():
    x = np.random.default_rng(5).standard_normal(700)
    sc = np.array([2.0, 5.0, 13.0, 40.0])
    W = B.blockwise_cwt(x, 300, 64, sc, fs=100.0)
    T, freqs = B.blockwise_ssq_cwt(x, 300, 64, sc, fs=100.0, maprange="maximal")
    assert W.shape == T.shape == (4, 700) and len(freqs) == 3
    e = B.extended_block(x, 300, 64, 2)  # the last block: 100 columns
    Wl, _, _ = O.cwt(e, scales=sc, fs=100.0)
    Tl, fl = O.ssq_cwt(e, scales=sc, fs=100.0, maprange="maximal")
    assert np.array_equal(W[:, 600:], Wl[:, 64:164]) and np.array_equal(T[:, 600:], Tl[:, 64:164])
    assert np.array_equal(freqs[2], fl) and not np.array_equal(freqs[0], fl)  # maximal: the block's own length
    # d = 0 and one block covering the recording: the whole-signal call
    Wf, _, _ = O.cwt(x, scales=sc, fs=100.0)
    assert np.array_equal(B.blockwise_cwt(x, 700, 0, sc, fs=100.0), Wf)

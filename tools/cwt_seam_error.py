"""Seam error of the blockwise CWT (the CWT stream, DESIGN §3.6b) against the whole-signal transform, in float64 on
the CPU (oracle/cwt_blocks.py against oracle/ssq_oracle.py): for each scale s and overlap d, the largest
|Wx_blocks - Wx_whole| over the interior blocks (all but the first and the last), relative to the largest |Wx_whole|
of that scale's row.  The first and last blocks are left out because there the two differ by construction: the
blocks mirror the recording with the edge sample repeated (dask's boundary="reflect"), the whole-signal call pads
without repeating it.  White noise, so every scale carries energy.  No GPU needed.

    python tools/cwt_seam_error.py [--wavelet gmw] [--n 32768] [--block 4096]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np  # noqa: E402

from oracle import cwt_blocks as B  # noqa: E402
from oracle import ssq_oracle as O  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--wavelet", default="gmw")
    ap.add_argument("--n", type=int, default=1 << 15)
    ap.add_argument("--block", type=int, default=1 << 12)
    ap.add_argument("--scales", default="4,16,64,256,1024")
    ap.add_argument("--overlaps", default="0,16,64,256,1024,4096")
    a = ap.parse_args()
    x = np.random.default_rng(0).standard_normal(a.n)
    sc = np.array([float(v) for v in a.scales.split(",")])
    ds = [int(v) for v in a.overlaps.split(",")]
    whole, _, _ = O.cwt(x, a.wavelet, sc)
    ref = np.abs(whole).max(axis=1)
    print(f"{a.wavelet}, N = {a.n}, block = {a.block}: interior max |Wx_blocks - Wx_whole| / max |Wx_whole| per scale")
    print("d \\ scale " + "".join(f"{s:>10g}" for s in sc))
    for d in ds:
        if d > a.block:
            continue
        W = B.blockwise_cwt(x, a.block, d, sc, wavelet=a.wavelet)
        inner = slice(a.block, a.n - a.block)
        err = np.abs(W[:, inner] - whole[:, inner]).max(axis=1) / ref
        print(f"{d:>9d} " + "".join(f"{e:>10.1e}" for e in err))


if __name__ == "__main__":
    main()

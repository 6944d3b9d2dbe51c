"""Upstream-compatible mode (SURVEY 8f rank 3): `stft`, `istft`, `ssq_stft`, `issq_stft` with the signatures, defaults
and conventions of upstream ssqueezepy (old/ssqueezepy/_stft.py:13-256, _ssq_stft.py:13-198), computed by the same CUDA
kernels as `ssqueeze._rs`.  What differs from the crate's conventions, and how it is obtained:

  * framing: upstream pads `n_fft // 2` samples on the left (the larger side for even n_fft, utils/common.py:116-120),
    the crate `(n_fft - 1) // 2` (stft_utils.rs:22) -> context option `upstream_framing`;
  * `modulated=True` by default (frames rotated by n_fft // 2, i.e. Sx[k] exp(+2 pi i k (n_fft // 2) / n_fft)): the
    library's SSQ_FLAG_MODULATED; upstream multiplies the derivative window by fs only when modulated
    (_stft.py:132-135), reproduced here;
  * windows: a string goes through scipy.signal.get_window(..., fftbins=True), None is dpss(win_len, win_len // 8),
    arrays are centre-padded to n_fft (utils/stft_utils.py get_window); n_fft defaults to min(N // hop_len, 512);
  * return values: `ssq_stft` -> (Tx, Sx, ssq_freqs, Sfs[, w][, dSx]), `stft` -> Sx (or (Sx, dSx)).

Arithmetic on the device is fp32 whatever `dtype` says (results come back as complex128 / float64).  `ssq_freqs`
other than the default grid, `flipud`, `t`, 2-D (batched) input and `astensor` are not supported here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import FLAG_MODULATED, PAD, SQUEEZE, Context, load, raise_status

__all__ = ["stft", "istft", "ssq_stft", "issq_stft", "get_window"]

_ctx = None


def _context():
    """A context of its own with upstream framing switched on (the default context keeps the crate's)."""
    global _ctx
    if _ctx is None:
        import os
        _ctx = Context(int(os.environ.get("SSQ_DEVICE", "0")))
        _ctx.set_option("upstream_framing", 1)
    return _ctx


def get_window(window, win_len, n_fft=None):
    """utils/stft_utils.py get_window: string -> scipy get_window (fftbins=True); None -> dpss(win_len, win_len // 8);
    array -> as is; then centre-padded to n_fft."""
    import scipy.signal as sig
    if n_fft is None:
        n_fft = win_len
    if window is None:
        w = sig.windows.dpss(win_len, max(4, win_len // 8), sym=False)
    elif isinstance(window, str):
        w = sig.get_window(window, win_len, fftbins=True)
    else:
        w = np.asarray(window, dtype=np.float64)
        if len(w) > n_fft:
            raise ValueError(f"len(window) = {len(w)} > n_fft = {n_fft}")
    w = np.asarray(w, dtype=np.float64)
    if len(w) < n_fft:
        pl = (n_fft - len(w)) // 2
        w = np.pad(w, [pl, n_fft - len(w) - pl])
    return np.ascontiguousarray(w)


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def _args(x, window, n_fft, win_len, hop_len):
    x = np.ascontiguousarray(x, dtype=np.float64)
    if x.ndim != 1:
        raise ValueError("compat mode takes 1-D input")
    N = len(x)
    n_fft = n_fft or min(N // hop_len, 512)
    if win_len is None:
        win_len = len(window) if isinstance(window, np.ndarray) else n_fft
    return x, N, int(n_fft), get_window(window, int(win_len), int(n_fft))


def stft(x, window=None, n_fft=None, win_len=None, hop_len=1, fs=None, t=None, padtype="reflect", modulated=True,
         derivative=False, dtype=None):
    """old/ssqueezepy/_stft.py:13-181."""
    Tx, Sx, _, _, dSx = ssq_stft(x, window, n_fft, win_len, hop_len, fs, t, modulated, padtype=padtype, get_dWx=True)
    return (Sx, dSx) if derivative else Sx


def ssq_stft(x, window=None, n_fft=None, win_len=None, hop_len=1, fs=None, t=None, modulated=True, ssq_freqs=None,
             padtype="reflect", squeezing="sum", gamma=None, preserve_transform=None, dtype=None, astensor=True,
             flipud=False, get_w=False, get_dWx=False):
    """old/ssqueezepy/_ssq_stft.py:13-136.  Returns (Tx, Sx, ssq_freqs, Sfs[, w][, dSx])."""
    if ssq_freqs is not None or flipud or t is not None:
        raise NotImplementedError("compat.ssq_stft: ssq_freqs / flipud / t are not supported")
    if padtype not in PAD:
        raise NotImplementedError(f"compat.ssq_stft: padtype {padtype!r} (reflect | zero)")
    x, N, n_fft, w = _args(x, window, n_fft, win_len, hop_len)
    fs = 1.0 if fs is None else float(fs)
    ctx = _context()
    nfq, nfr = n_fft // 2 + 1, (N - 1) // hop_len + 1
    Tx = np.empty((nfq, nfr), dtype=np.complex128)
    Sx = np.empty((nfq, nfr), dtype=np.complex128)
    dSx = np.empty((nfq, nfr), dtype=np.complex128)
    wph = np.empty((nfq, nfr), dtype=np.float64)
    sf = np.empty(nfq, dtype=np.float64)
    # upstream applies `* fs` to the derivative window only inside `if modulated:` (_stft.py:132-135)
    fs_eff = fs if modulated else 1.0
    g = float("nan") if gamma is None else float(gamma)
    st = load().ssq_ssq_stft_f64(ctx.handle, _ptr(x), N, _ptr(w), len(w), n_fft, len(w), int(hop_len), fs_eff,
                                 PAD[padtype], SQUEEZE.get(squeezing, 0), g, FLAG_MODULATED if modulated else 0, _ptr(Tx),
                                 _ptr(sf), _ptr(Sx), _ptr(dSx), _ptr(wph), C.c_void_p(0))
    raise_status(st, ctx.handle)
    Sfs = np.linspace(0, 0.5 * fs, nfq)
    if not modulated and fs != 1.0:
        # the kernel ran with fs = 1: its w and grid are in cycles/sample, upstream's Sfs in Hz with an unscaled dSx
        raise NotImplementedError("compat.ssq_stft: modulated=False with fs != 1 (upstream mixes units there)")
    out = [Tx, Sx, Sfs.copy(), Sfs]
    if get_w:
        out.append(wph)
    if get_dWx:
        out.append(dSx)
    return tuple(out)


def istft(Sx, window=None, n_fft=None, win_len=None, hop_len=1, N=None, modulated=True, win_exp=1):
    """old/ssqueezepy/_stft.py:184-256."""
    Sx = np.ascontiguousarray(Sx, dtype=np.complex128)
    nfq, nfr = Sx.shape
    n_fft = n_fft or (nfq - 1) * 2
    win_len = win_len or (len(window) if isinstance(window, np.ndarray) else n_fft)
    N = N or hop_len * nfr
    w = get_window(window, int(win_len), int(n_fft))
    if modulated:  # undo the rotation of the frames: Sx[k] exp(-2 pi i k (n_fft // 2) / n_fft)
        k = np.arange(nfq)
        Sx = Sx * np.exp(-2j * np.pi * k * (n_fft // 2) / n_fft)[:, None]
        Sx = np.ascontiguousarray(Sx)
    ctx = _context()
    x = np.empty(int(N), dtype=np.float64)
    st = load().ssq_istft_f64(ctx.handle, _ptr(Sx), nfq, nfr, _ptr(w), len(w), int(n_fft), int(hop_len), int(N),
                              int(win_exp), _ptr(x))
    raise_status(st, ctx.handle)
    return x


def issq_stft(Tx, window=None, cc=None, cw=None, n_fft=None, win_len=None, hop_len=1, modulated=True):
    """old/ssqueezepy/_ssq_stft.py:139-198.  Without `cc` / `cw` the full inversion, [n_frames]; with them the curve
    bands of `_invert_components` (_ssq_cwt.py:380-402) times upstream's 2 / window[n_fft // 2], [K + 1, n_frames]
    with the residual last.  1-D cc / cw are one band, as upstream's reshape(-1, 1)."""
    if not modulated:
        raise ValueError("inversion with `modulated == False` is unsupported.")
    if hop_len != 1:
        raise ValueError("inversion with `hop_len != 1` is unsupported.")
    if (cc is None) != (cw is None):
        raise ValueError("cc and cw go together")
    Tx = np.ascontiguousarray(Tx, dtype=np.complex128)
    nfq, nfr = Tx.shape
    n_fft = n_fft or (nfq - 1) * 2
    win_len = win_len or n_fft
    if cc is not None:
        cc, cw = np.asarray(cc), np.asarray(cw)
        cc, cw = (cc.reshape(-1, 1) if cc.ndim == 1 else cc), (cw.reshape(-1, 1) if cw.ndim == 1 else cw)
        if cc.ndim != 2 or cc.shape != cw.shape or cc.shape[0] != nfr:
            raise ValueError(f"cc {cc.shape} and cw {cw.shape} must both be [n_frames = {nfr}, K]")
        cc = np.ascontiguousarray(cc, dtype=np.int32)
        cw = np.ascontiguousarray(cw, dtype=np.int32)
        w = get_window(window, int(win_len), int(n_fft))
        ctx = _context()
        y = np.empty((cc.shape[1] + 1, nfr), dtype=np.float64)
        st = load().ssq_issq_stft_components_f64(ctx.handle, _ptr(Tx), nfq, nfr, _ptr(w), len(w), int(n_fft), 1, 1.0,
                                                 _ptr(cc), _ptr(cw), cc.shape[1], _ptr(y))
        raise_status(st, ctx.handle)
        return y
    w = get_window(window, int(win_len), int(n_fft))
    ctx = _context()
    y = np.empty(nfr, dtype=np.float64)
    st = load().ssq_issq_stft_f64(ctx.handle, _ptr(Tx), nfq, nfr, _ptr(w), len(w), int(n_fft), 1, 1.0, _ptr(y))
    raise_status(st, ctx.handle)
    return y

"""CPU oracle for the ssqueeze._rs hot path -- TEST INFRASTRUCTURE, NOT PRODUCT.

A float64 NumPy restatement of the reference's Rust transforms
(`/root/reference/rust/src/spectral/*.rs`).  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this module; the product path (`ssqueeze_rs_b200`) never does.

Parity pin status
-----------------
The reference cannot be built here (no rustc/cargo, crates not vendored) and
its own tests hold no golden vectors (they print shapes only), so parity
against the Rust binary itself is UNPINNED.  What *is* pinned:

* the restatement agrees with the vendored upstream `old/ssqueezepy`
  (imported in the build container) wherever the two implementations must
  coincide -- vectors committed by `tests/golden/make_golden.py`:
  odd n_fft, fs=1, modulated=False (`upstream_odd.npz`: Sx, dSx, Tx, istft to
  1e-12); the BENCHMARK geometry n_fft=512, hop=32 on every frame that touches
  no padding, via upstream run on the one-sample-shifted signal
  (`upstream_even512.npz`: 4e-16); the CWT core and phase transform
  (`upstream_cwt.npz`: all gmw rows 3e-15, morlet rows away from Nyquist 1e-8);
  the admissibility constants (`upstream_adm.npz`);
* every shape/dtype expectation of the reference smoke scripts
  (`tests/stft_test.py:137-151`, `tests/stft_ssq_test.py:132-152`,
  `tests/cwt_test.py:19-57`, `tests/ssq_cwt_test.py:19-57,410-419`).

Third-party arithmetic absent from /root/reference: all FFTs are
`rustfft = "6.2.0"` (rust/Cargo.toml:15-27): unnormalised forward
exp(-2*pi*i*k*n/N), unnormalised inverse.  Any correct f64 DFT agrees to
~1e-15 relative; numpy's pocketfft is used here.

Each function cites the reference file:line it follows.
"""
from __future__ import annotations

import math
import numpy as np

EPS64 = 2.2204460492503131e-16
TWO_PI_LITERAL = 6.283185307179586  # ssq_stft.rs:32


# --------------------------------------------------------------------------
# STFT-side helpers
# --------------------------------------------------------------------------
def pad_reflect_stft(x: np.ndarray, n_fft: int) -> np.ndarray:
    """stft_utils.rs:19-49.  Total pad n_fft-1, left=(n_fft-1)//2 (the smaller
    side for even n_fft); numpy-'reflect' style (no edge repeat); where the
    mirror index runs outside x the sample stays zero (guards at :35, :43 --
    usize wrap-around in release builds makes the right guard a no-op skip)."""
    n = len(x)
    pad = n_fft - 1
    left = pad // 2
    right = pad - left
    out = np.zeros(n + pad, dtype=np.float64)
    out[left:left + n] = x
    i = np.arange(left)
    m = left - i
    ok = m < n
    out[i[ok]] = x[m[ok]]
    i = np.arange(right)
    m = n - 2 - i
    ok = (m >= 0) & (m < n)
    out[n + left + i[ok]] = x[m[ok]]
    return out


def pad_zeros_stft(x: np.ndarray, n_fft: int) -> np.ndarray:
    """stft_utils.rs:52-65."""
    n = len(x)
    pad = n_fft - 1
    left = pad // 2
    out = np.zeros(n + pad, dtype=np.float64)
    out[left:left + n] = x
    return out


def pad_upstream_stft(x: np.ndarray, n_fft: int, padtype: str) -> np.ndarray:
    """Upstream ssqueezepy's framing (old/ssqueezepy/utils/common.py:116-120, padsignal): left n_fft//2 (the larger
    side for even n_fft), right n_fft-1-n_fft//2, by np.pad.  'reflect' reflects again and again where a pad is longer
    than the signal (N <= n_fft//2), and a 1-sample signal becomes a constant; 'zero' pads zeros."""
    left = n_fft // 2
    return np.pad(x, [left, n_fft - 1 - left], mode="constant" if padtype == "zero" else "reflect")


def _pad_stft(x, n_fft, padtype, framing="crate"):
    # stft.rs:25-29 / ssq_stft.rs:124-128: unknown strings fall back to reflect
    if framing == "upstream":
        return pad_upstream_stft(x, n_fft, padtype)
    if framing != "crate":
        raise ValueError(f"framing must be 'crate' or 'upstream', not {framing!r}")
    if padtype == "zero":
        return pad_zeros_stft(x, n_fft)
    return pad_reflect_stft(x, n_fft)


def pad_left(n_fft: int, framing: str = "crate") -> int:
    """Left pad of a framing: frame f starts at sample f*hop - pad_left, and `istft` unpads there."""
    if framing not in ("crate", "upstream"):
        raise ValueError(f"framing must be 'crate' or 'upstream', not {framing!r}")
    return n_fft // 2 if framing == "upstream" else (n_fft - 1) // 2


def _frames(padded: np.ndarray, n_fft: int, hop: int) -> np.ndarray:
    """[n_frames, n_fft] view of the padded signal (stft.rs:32-33, 51-55)."""
    n_frames = (len(padded) - n_fft) // hop + 1
    idx = np.arange(n_frames)[:, None] * hop + np.arange(n_fft)[None, :]
    return padded[idx]


def stft(x, n_fft, hop_length, window, padtype, *, framing="crate"):
    """stft.rs:12-95.  Returns (Sx complex128 [n_fft//2+1, n_frames],
    freqs = linspace(0, 0.5, n_freqs)).  The window is NOT resized: a window
    longer than n_fft is truncated to its first n_fft taps
    (stft_utils.rs:8), a shorter one makes rustfft panic.  framing="upstream"
    pads as upstream ssqueezepy does (`pad_upstream_stft`)."""
    x = np.asarray(x, dtype=np.float64)
    window = np.asarray(window, dtype=np.float64)
    if hop_length < 1:
        raise ZeroDivisionError("hop_length must be >= 1 (stft.rs:33 divides by it)")
    if len(window) < n_fft:
        raise RuntimeError("window shorter than n_fft: rustfft buffer-length panic "
                           "(stft_utils.rs:8, stft.rs:67)")
    if len(x) < 1:
        raise RuntimeError("empty x: usize underflow at stft.rs:33")
    padded = _pad_stft(x, n_fft, padtype, framing)
    fr = _frames(padded, n_fft, hop_length) * window[:n_fft][None, :]
    n_freqs = n_fft // 2 + 1
    Sx = np.fft.fft(fr, axis=1)[:, :n_freqs].T.copy()
    freqs = np.linspace(0.0, 0.5, n_freqs)
    return Sx, freqs


def fit_window(window: np.ndarray, n_fft: int) -> np.ndarray:
    """ssq_stft.rs:104-119: centre zero-pad (left=(n_fft-len)//2) or centre
    crop (start=(len-n_fft)//2)."""
    window = np.asarray(window, dtype=np.float64)
    L = len(window)
    if L < n_fft:
        left = (n_fft - L) // 2
        out = np.zeros(n_fft, dtype=np.float64)
        out[left:left + L] = window
        return out
    if L > n_fft:
        start = (L - n_fft) // 2
        return window[start:start + n_fft].copy()
    return window.copy()


def diff_window(window_sized: np.ndarray) -> np.ndarray:
    """ssq_stft.rs:131-179: Re(IFFT(FFT(w) * i*xi)) / n with
    xi_k = 2*pi*k/n for k <= n/2 (Nyquist POSITIVE), 2*pi*(k-n)/n above."""
    n = len(window_sized)
    k = np.arange(n, dtype=np.float64)
    k[n // 2 + 1:] -= n
    xi = k * (2.0 * math.pi / n)
    W = np.fft.fft(window_sized)
    W = (-W.imag * xi) + 1j * (W.real * xi)
    return (np.fft.ifft(W) * n).real * (1.0 / n)


def ssq_freqs_stft(n_freqs: int, fs: float) -> np.ndarray:
    """ssq_stft.rs:42-54."""
    i = np.arange(n_freqs, dtype=np.float64)
    return i * 0.5 * fs / (float(n_freqs) - 1.0)


def phase_stft(Sx, dSx, Sfs, gamma):
    """ssq_stft.rs:11-39.  |Sx| < gamma -> +inf, else
    |Sfs[i] - (b*c - a*d) / ((c*c + d*d) * 2pi)|."""
    a, b = dSx.real, dSx.imag
    c, d = Sx.real, Sx.imag
    with np.errstate(all="ignore"):
        pd = (b * c - a * d) / ((c * c + d * d) * TWO_PI_LITERAL)
        w = np.abs(Sfs[:, None] - pd)
    w[np.hypot(c, d) < gamma] = np.inf
    return w


def reassign_stft(Sx, w, ssq_freqs, squeezing):
    """ssq_stft.rs:270-301.  Literal arg-min over the whole grid with strict
    '<' (ties -> lower index, out of range clamps, NaN -> bin 0); weights
    accumulated in ascending source-row order; each contribution times
    dw = ssq_freqs[1]-ssq_freqs[0]."""
    n_freqs, n_frames = Sx.shape
    dw = ssq_freqs[1] - ssq_freqs[0]
    Tx = np.zeros((n_freqs, n_frames), dtype=np.complex128)
    kk = np.full((n_freqs, n_frames), -1, dtype=np.int64)
    cols = np.arange(n_frames)
    leb = complex(1.0 / float(n_freqs), 0.0)
    chunk = max(1, (1 << 22) // max(1, n_freqs))
    for i in range(n_freqs):
        wi = w[i]
        fin = ~np.isinf(wi)
        k = np.zeros(n_frames, dtype=np.int64)
        for s in range(0, n_frames, chunk):
            with np.errstate(invalid="ignore"):
                dist = np.abs(wi[s:s + chunk, None] - ssq_freqs[None, :])
            # NaN rows: every comparison `dist < min_dist` is false -> k = 0
            nanrow = np.isnan(wi[s:s + chunk])
            dist[nanrow, :] = 0.0
            k[s:s + chunk] = np.argmin(dist, axis=1)
        weight = Sx[i] if squeezing != "lebesgue" else np.full(n_frames, leb)
        sel = cols[fin]
        Tx[k[fin], sel] += weight[fin] * dw
        kk[i, fin] = k[fin]
    return Tx, kk


def ssq_stft(x, window, n_fft=None, win_len=None, hop_len=1, fs=1.0,
             padtype="reflect", squeezing="sum", gamma=None, *,
             modulated=False, return_aux=False, framing="crate"):
    """ssq_stft.rs:74-313.  `modulated` / `return_aux` / `framing` are build-side
    extensions (SURVEY 8a row 10, 8b): modulated multiplies Sx and dSx rows by
    exp(+2*pi*i*k*(n_fft//2)/n_fft) before squeezing (w is unaffected);
    framing="upstream" pads as upstream ssqueezepy does (`pad_upstream_stft`)."""
    x = np.asarray(x, dtype=np.float64)
    window = np.asarray(window, dtype=np.float64)
    n = len(x)
    n_fft = n_fft if n_fft is not None else min(n, 512)
    win_len = win_len if win_len is not None else len(window)
    if win_len > n_fft:
        raise ValueError(f"Window length {win_len} cannot be greater than n_fft {n_fft}")
    if hop_len < 1:
        raise ZeroDivisionError("hop_len must be >= 1 (ssq_stft.rs:183)")
    if n < 1:
        raise RuntimeError("empty x: usize underflow at ssq_stft.rs:183")
    wsz = fit_window(window, n_fft)
    padded = _pad_stft(x, n_fft, padtype, framing)
    dwin = diff_window(wsz)
    fr = _frames(padded, n_fft, hop_len)
    n_freqs = n_fft // 2 + 1
    Sx = np.fft.fft(fr * wsz[None, :], axis=1)[:, :n_freqs].T.copy()
    dSx = np.fft.fft(fr * dwin[None, :] * fs, axis=1)[:, :n_freqs].T.copy()
    if modulated:
        ph = np.exp(2j * math.pi * np.arange(n_freqs) * (n_fft // 2) / n_fft)
        Sx = Sx * ph[:, None]
        dSx = dSx * ph[:, None]
    Sfs = np.linspace(0.0, 0.5 * fs, n_freqs)
    g = gamma if gamma is not None else 10.0 * EPS64
    w = phase_stft(Sx, dSx, Sfs, g)
    sf = ssq_freqs_stft(n_freqs, fs)
    Tx, kk = reassign_stft(Sx, w, sf, squeezing)
    if return_aux:
        return Tx, sf, dict(Sx=Sx, dSx=dSx, w=w, k=kk, window=wsz, diff_window=dwin)
    return Tx, sf


def istft(Sx, window, n_fft=None, win_len=None, hop_len=1, N=None, win_exp=1, *, framing="crate"):
    """Inverse of `stft` in the Rust framing convention.  Absent from the Rust
    crate (lib.rs:25-32); specified from old/ssqueezepy/_stft.py:184-256 and
    old/ssqueezepy/utils/stft_utils.py:141-191 with modulated=False, and the
    Rust pad offset (n_fft-1)//2 (stft_utils.rs:22) for unpadding, or
    upstream's n_fft//2 with framing="upstream"."""
    Sx = np.asarray(Sx)
    n_fft = n_fft or (Sx.shape[0] - 1) * 2
    left = pad_left(n_fft, framing)
    n_frames = Sx.shape[1]
    N = N or hop_len * n_frames
    wsz = fit_window(window, n_fft)
    xbuf = np.fft.irfft(Sx, n=n_fft, axis=0)
    wa = np.ones(n_fft) if win_exp == 0 else wsz ** win_exp
    L = N + n_fft - 1
    xr = np.zeros(L, dtype=np.float64)
    for j in range(n_frames):
        s = j * hop_len
        if s + n_fft > L:
            break
        xr[s:s + n_fft] += xbuf[:, j] * wa
    wn = np.zeros(L, dtype=np.float64)
    wpow = wsz ** (win_exp + 1)
    for j in range((L - n_fft) // hop_len + 1):
        s = j * hop_len
        wn[s:s + n_fft] += wpow
    tiny = np.finfo(np.float64).tiny
    nz = wn > tiny
    xr[nz] /= wn[nz]
    return xr[left:left + N]


def issq_stft(Tx, window, n_fft=None, win_len=None, hop_len=1, fs=1.0):
    """old/ssqueezepy/_ssq_stft.py:139-198 (full inverse):
    x[j] = sum_k Re Tx[k, j] * 2 / w[n_fft//2]; the Rust Tx carries an extra
    dw = fs/n_fft factor relative to upstream at fs=1 (ssq_stft.rs:273,298), so
    the result is divided by fs.  Needs hop_len == 1 and Tx from a *modulated*
    transform.  y[j] estimates padded sample j + n_fft//2, i.e.
    x[j + n_fft//2 - (n_fft-1)//2]."""
    if hop_len != 1:
        raise ValueError("inversion with `hop_len != 1` is unsupported.")
    Tx = np.asarray(Tx)
    n_fft = n_fft or (Tx.shape[0] - 1) * 2
    wsz = fit_window(window, n_fft)
    y = Tx.real.sum(axis=0)
    return y * (2.0 / wsz[n_fft // 2]) / fs


# --------------------------------------------------------------------------
# CWT side
# --------------------------------------------------------------------------
def next_power_of_2(n: int) -> int:
    """utils/array.rs:9-11: 1 << ceil(log2(n)) via f64."""
    if n <= 0:
        return 1
    return 1 << int(math.ceil(math.log2(float(n))))


def pad_reflect_cwt(x, pad_len):
    """utils/array.rs:52-82."""
    n = len(x)
    pad = pad_len - n
    left = pad // 2
    right = pad - left
    out = np.zeros(pad_len, dtype=np.float64)
    out[left:left + n] = x
    i = np.arange(left)
    m = left - i
    ok = m < n
    out[i[ok]] = x[m[ok]]
    i = np.arange(right)
    m = n - 2 - i
    ok = (m >= 0) & (m < n)
    out[n + left + i[ok]] = x[m[ok]]
    return out


def pad_zero_cwt(x, pad_len):
    """utils/array.rs:85-98."""
    n = len(x)
    left = (pad_len - n) // 2
    out = np.zeros(pad_len, dtype=np.float64)
    out[left:left + n] = x
    return out


def xifn(scale: float, n: int) -> np.ndarray:
    """wavelets/base.rs:18-33 (Nyquist bin positive)."""
    h = scale * (2.0 * math.pi) / float(n)
    k = np.arange(n, dtype=np.float64)
    k[n // 2 + 1:] -= n
    return k * h


def generate_wavelet_fourier(xi, scale, wavelet):
    """cwt.rs:492-547.  'morlet' (w >= 0): pi^-1/4*sqrt2*(exp(-(w-6)^2/2) -
    exp(-18)*exp(-w^2/2)); anything else = GMW gamma=3, beta=60 (w > 0):
    2*exp(60 ln w - w^3), not peak-normalised."""
    w = scale * xi
    out = np.zeros(len(xi), dtype=np.float64)
    if wavelet == "morlet":
        mu = 6.0
        norm = math.pi ** (-0.25) * math.sqrt(2.0)
        k_exp = math.exp(-0.5 * mu * mu)
        pos = w >= 0.0
        wp = w[pos]
        out[pos] = norm * (np.exp(-0.5 * (wp - mu) ** 2) - k_exp * np.exp(-0.5 * wp ** 2))
    else:
        pos = w > 0.0
        wp = w[pos]
        out[pos] = 2.0 * np.exp(60.0 * np.log(wp) - wp ** 3.0)
    return out


def generate_log_scales(N, nv, simd=False):
    """cwt.rs:461-489 (2^p) and cwt_simd.rs:474-545 (exp(p*ln2) when >= 16
    scales)."""
    log_min = math.log2(2.0)
    log_max = math.log2(float(N) * 0.5)
    ns = int(math.ceil((log_max - log_min) * float(nv)))
    sf = (log_max - log_min) / float(ns - 1) if ns > 1 else 0.0
    p = log_min + np.arange(ns, dtype=np.float64) * sf
    if simd and ns >= 16:
        return np.exp(p * math.log(2.0))
    return np.power(2.0, p)


def _dt(fs, t):
    if t is not None:
        t = np.asarray(t, dtype=np.float64)
        if len(t) < 2:
            raise ValueError("Time vector must have at least 2 elements")
        return float(t[1] - t[0])
    if fs is not None:
        return 1.0 / float(fs)
    return 1.0


def _cwt_core(x, wavelet, scales, dt, padtype, derivative):
    """cwt.rs:85-96 + 169-326 / ssq_cwt.rs:331-431 (padded rows)."""
    N = len(x)
    pad_len = next_power_of_2(N + N // 2)
    padded = pad_zero_cwt(x, pad_len) if padtype == "zero" else pad_reflect_cwt(x, pad_len)
    xh = np.fft.fft(padded)
    xi = xifn(1.0, pad_len)
    ns = len(scales)
    Wx = np.empty((ns, pad_len), dtype=np.complex128)
    dWx = np.empty((ns, pad_len), dtype=np.complex128) if derivative else None
    inv = 1.0 / float(pad_len)
    for i, s in enumerate(scales):
        psih = generate_wavelet_fourier(xi, s, wavelet)
        Wx[i] = (np.fft.ifft(xh * psih) * pad_len) * inv
        if derivative:
            dpsih = psih * (1j * (xi / dt))
            dWx[i] = (np.fft.ifft(xh * dpsih) * pad_len) * inv
    n1 = (pad_len - N) // 2
    return Wx, dWx, n1, pad_len


def cwt(x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=True,
        derivative=False, padtype="reflect", rpadded=False, vectorized=True,
        patience=0, *, _simd=False):
    """cwt.rs:46-144.  Always a 3-tuple (Wx, scales, dWx|None)."""
    x = np.asarray(x, dtype=np.float64)
    N = len(x)
    dt = _dt(fs, t)
    scales = (np.asarray(scales, dtype=np.float64).copy() if scales is not None
              else generate_log_scales(N, nv, simd=_simd))
    Wx, dWx, n1, pad_len = _cwt_core(x, wavelet, scales, dt, padtype, derivative)
    if not l1_norm:
        f = np.sqrt(scales)[:, None]  # cwt.rs:253
        Wx = Wx * f
        if dWx is not None:
            dWx = dWx * f
    if not rpadded:
        Wx = Wx[:, n1:n1 + N].copy()
        if dWx is not None:
            dWx = dWx[:, n1:n1 + N].copy()
    return Wx, scales, dWx


def cwt_simd(*args, **kwargs):
    """cwt_simd.rs:52-614: same numbers as `cwt` except the default-scale
    generator (exp(p ln2) for >= 16 scales)."""
    return cwt(*args, _simd=True, **kwargs)


def phase_cwt(Wx, dWx, gamma):
    """ssq_cwt.rs:15-47."""
    a, b = dWx.real, dWx.imag
    c, d = Wx.real, Wx.imag
    with np.errstate(all="ignore"):
        w = np.abs((b * c - a * d) / ((c * c + d * d) * 2.0 * math.pi))
    w[np.hypot(c, d) < gamma] = np.inf
    return w


def ssq_freqs_cwt(n_freqs, fmin, fmax, distribution):
    """ssq_cwt.rs:50-113 ('linear', else log2-spaced)."""
    i = np.arange(n_freqs, dtype=np.float64)
    if distribution == "linear":
        step = (fmax - fmin) / float(n_freqs - 1) if n_freqs > 1 else 0.0
        return fmin + i * step
    lmin, lmax = math.log2(fmin), math.log2(fmax)
    sf = (lmax - lmin) / float(n_freqs - 1) if n_freqs > 1 else 0.0
    return np.power(2.0, lmin + i * sf)


def _round_half_away(v):
    return np.sign(v) * np.floor(np.abs(v) + 0.5)


def ssqueeze_cwt(Wx, w, ssq_freqs, squeezing, flipud):
    """ssq_cwt.rs:116-222.  is_log := f[1]/f[0] > 1.1; closed-form bin with
    f64::round (half away from zero); out-of-range / inf / NaN dropped;
    k = ns-1-bin when flipud; Tx[k, j] += Wx[i, j] or 1/n_scales."""
    ns, nt = Wx.shape
    nf = len(ssq_freqs)
    Tx = np.zeros((nf, nt), dtype=np.complex128)
    kk = np.full((ns, nt), -1, dtype=np.int64)
    is_log = (ssq_freqs[1] / ssq_freqs[0] > 1.1) if nf > 1 else False
    if is_log:
        lmin = math.log2(ssq_freqs[0])
        lstep = (math.log2(ssq_freqs[nf - 1]) - lmin) / float(nf - 1) if nf > 1 else 1.0
    else:
        lin_min = ssq_freqs[0]
        lin_step = (ssq_freqs[nf - 1] - lin_min) / float(nf - 1) if nf > 1 else 1.0
    cols = np.arange(nt)
    leb = complex(1.0 / float(ns), 0.0)
    for i in range(ns):
        wi = w[i]
        ok = np.isfinite(wi)
        with np.errstate(all="ignore"):
            if is_log:
                b = _round_half_away((np.log2(wi) - lmin) / lstep)
            else:
                b = _round_half_away((wi - lin_min) / lin_step)
        # `as isize` saturates (+-inf -> isize::MIN/MAX, both out of range)
        b = np.where(np.isfinite(b), b, -1.0)
        b = np.clip(b, -2.0 ** 62, 2.0 ** 62).astype(np.int64)
        ok &= (b >= 0) & (b < nf)
        k = (nf - 1 - b) if flipud else b
        weight = Wx[i] if squeezing != "lebesgue" else np.full(nt, leb)
        Tx[k[ok], cols[ok]] += weight[ok]
        kk[i, ok] = k[ok]
    return Tx, kk


def ssq_cwt(x, wavelet="gmw", scales=None, fs=None, t=None, ssq_freqs=None, nv=32,
            padtype="reflect", squeezing="sum", maprange="peak", difftype="trig",
            gamma=None, vectorized=True, flipud=True, *, return_aux=False):
    """ssq_cwt.rs:261-493.  `difftype` and `vectorized` are ignored
    (:296-297)."""
    x = np.asarray(x, dtype=np.float64)
    N = len(x)
    dt = _dt(fs, t)
    scales = (np.asarray(scales, dtype=np.float64).copy() if scales is not None
              else generate_log_scales(N, nv, simd=False))
    Wx, dWx, n1, pad_len = _cwt_core(x, wavelet, scales, dt, padtype, True)
    Wx = Wx[:, n1:n1 + N]
    dWx = dWx[:, n1:n1 + N]
    g = gamma if gamma is not None else 10.0 * EPS64
    w = phase_cwt(Wx, dWx, g)
    dist = ssq_freqs if ssq_freqs is not None else "log"
    if maprange == "maximal":
        dT = float(N) * dt
        fmin, fmax = 1.0 / dT, 0.5 / dt
    else:
        fmin, fmax = 1.0 / scales[-1], 1.0 / scales[0]
    sf = ssq_freqs_cwt(len(scales), fmin, fmax, dist)
    Tx, kk = ssqueeze_cwt(Wx, w, sf, squeezing, flipud)
    if return_aux:
        return Tx, sf, dict(Wx=Wx, dWx=dWx, w=w, k=kk, scales=scales)
    return Tx, sf


# --------------------------------------------------------------------------
# icwt (SURVEY 8f rank 2; cwt.rs:548-718, a #[pyfunction] the module never registers)
# --------------------------------------------------------------------------
def adm_ssq(wavelet="gmw"):
    """Css = integral_0^inf psi-hat(w)/w dw (old/ssqueezepy/utils/cwt_utils.py:28-47) of the wavelet
    generate_wavelet_fourier evaluates (cwt.rs:492-547), by adaptive quadrature."""
    from scipy.integrate import quad
    one = np.ones(1)
    f = lambda w: float(generate_wavelet_fourier(one * w, 1.0, wavelet)[0].real) / w
    pts = [6.0] if wavelet == "morlet" else [20.0 ** (1.0 / 3.0)]
    return quad(f, 1e-12, 60.0, points=pts, epsabs=0.0, epsrel=1e-13, limit=2000)[0]


def invert_components(Tx, cc, cw):
    """old/ssqueezepy/_ssq_cwt.py:380-402, restated: per component the rows cc-cw .. cc+cw of every column
    (clipped to [0, n_rows]; cc == -1: none), each from the original Tx; last row: what no band covers."""
    Tx = np.asarray(Tx)
    n_rows, n = Tx.shape
    cc = np.asarray(cc).reshape(n, -1).astype(np.int64)
    cw = np.asarray(cw).reshape(n, -1).astype(np.int64)
    K = cc.shape[1]
    x = np.zeros((K + 1, n))
    rest = Tx.real.copy()
    for c in range(K):
        upper = np.clip(cc[:, c] + cw[:, c], 0, n_rows)
        lower = np.clip(cc[:, c] - cw[:, c], 0, n_rows)
        upper[cc[:, c] == -1] = 0
        lower[cc[:, c] == -1] = 1
        for m in range(n):
            sl = slice(lower[m], upper[m] + 1)
            x[c, m] = Tx.real[sl, m].sum()
            rest[sl, m] = 0.0
    x[K] = rest.sum(axis=0)
    return x


def issq_cwt(Tx, wavelet="gmw", scales=None, cc=None, cw=None):
    """old/ssqueezepy/_ssq_cwt.py:313-378 in the reference's framing: the log-step `const` upstream bakes into
    Tx is applied here (the reference's ssqueeze omits it, ssq_cwt.rs:116-222)."""
    Tx = np.asarray(Tx, dtype=np.complex128)
    if scales is None:
        raise ValueError("Scales must be provided")
    scales = np.asarray(scales, dtype=np.float64)
    dj = math.log(scales[1] / scales[0]) if (len(scales) > 1 and scales[1] > scales[0]) else 0.1
    if cc is not None:
        return invert_components(Tx, cc, cw) * (2.0 / adm_ssq(wavelet)) * dj
    x = np.zeros(Tx.shape[1])
    for i in range(Tx.shape[0]):
        x += Tx[i].real
    return x * (2.0 / adm_ssq(wavelet)) * dj


def icwt(Wx, wavelet="gmw", scales=None, nv=None, one_int=True, x_len=None, x_mean=0.0,
         padtype="reflect", rpadded=False, l1_norm=True, exact_adm=False):
    """cwt.rs:548-718: the one-integral branch (:590-627, the default) and the two-integral branch (:629-712;
    the device builds the latter for power-of-two x_len == Wx.shape[1] only)."""
    Wx = np.asarray(Wx, dtype=np.complex128)
    if scales is None:
        raise ValueError("Scales must be provided")  # cwt.rs:572-575
    scales = np.asarray(scales, dtype=np.float64)
    n_scales, n_times = Wx.shape
    adm = 0.776 if wavelet == "morlet" else 1.0       # cwt.rs:579-583
    if exact_adm:
        adm = adm_ssq(wavelet)
    x_length = n_times if x_len is None else int(x_len)
    if x_length > n_times:
        raise IndexError("x_len > Wx.shape[1]: ndarray index out of bounds (panic) at cwt.rs:613")
    if not one_int:
        # cwt.rs:629-712: per scale FFT(Wx[i, :x_len]) * conj(psi-hat(scale xi)) -> IFFT; real part / x_len times
        # 1/scale (l1) or 1/sqrt(scale)^2 (otherwise: the same number); summed, then * (2/adm) dj + x_mean
        xi = xifn(1.0, x_length)
        x = np.zeros(x_length)
        for i in range(n_scales):
            psih = generate_wavelet_fourier(xi, scales[i], wavelet)
            tmp = np.fft.ifft(np.fft.fft(Wx[i, :x_length]) * np.conj(psih)) * x_length  # rustfft: unnormalised inverse
            scale_norm = 1.0 / scales[i] if l1_norm else 1.0 / math.sqrt(scales[i]) ** 2
            x += tmp.real * (1.0 / x_length) * scale_norm
        dj = math.log(scales[1] / scales[0]) if (n_scales > 1 and scales[1] > scales[0]) else 0.1
        return x * ((2.0 / adm) * dj) + x_mean
    dj = math.log(scales[1] / scales[0]) if (n_scales > 1 and scales[1] > scales[0]) else 0.1  # :595-599
    final_norm = (2.0 / adm) * dj
    norm = np.ones(n_scales) if l1_norm else 1.0 / np.sqrt(scales[:n_scales])                 # :606-610
    x = np.zeros(x_length)
    for i in range(n_scales):                                                                  # :620-623 (i ascending)
        x += Wx[i, :x_length].real * norm[i]
    return x * final_norm + x_mean                                                             # :624

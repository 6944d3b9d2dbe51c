"""Host-side mirror of the reference's `ssqueeze._rs` module (rust/src/lib.rs:23-35):
same callables, argument order, defaults, dtypes, return arity and error
behaviour, each forwarding to one C-ABI call of libssqcuda (include/ssqcuda.h).

The reference host layer is Rust/pyo3; no Rust toolchain exists in this image,
so this module plays that role (INTEGRATION.md holds the pyo3 source a
maintainer would compile instead).  Inputs must be 1-D float64 numpy arrays,
as `PyReadonlyArray1<f64>` demands (anything else -> TypeError); outputs are
freshly allocated C-contiguous complex128 / float64 arrays.

Additions over the reference (north star): `istft`, `issq_stft`, the
keyword-only extras `modulated=` / `return_aux=` of `ssq_stft`, and
`ssq_stft_batch` -- all channels of a recording in one call (the per-channel
loop of the reference's tests/stft_ssq_test.py:230-251), complex64 out, pinned
host memory or the device: the scalar call spends its time converting to
float64 / complex128 (12.5 ms per 1.8 M-sample channel for 0.1 ms of kernel).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (FLAG_ADM_EXACT, FLAG_L2_NORM, FLAG_MODULATED, FLAG_NO_FLIPUD, FLAG_RPADDED, FLAG_SIMD_SCALES, PAD, SQUEEZE,
                   default_context, load, raise_status)

__all__ = ["hello_from_bin", "stft", "stft_batch", "ssq_stft", "ssq_stft_batch", "ssq_cwt_batch", "pinned_empty", "istft", "issq_stft", "cwt", "cwt_simd", "ssq_cwt", "icwt", "issq_cwt",
           "adm_ssq", "extract_ridges", "morlet", "morlet_freq", "morlet_time", "gmw", "gmw_freq", "gmw_time",
           "gmw_center_frequency"]


def _f64_1d(a, name):
    # PyReadonlyArray1<f64>: must already be a float64 ndarray of rank 1
    if not isinstance(a, np.ndarray) or a.dtype != np.float64 or a.ndim != 1:
        raise TypeError(f"argument '{name}': expected a 1-D numpy.ndarray of float64, got "
                        f"{type(a).__name__}" + (f" dtype={a.dtype} ndim={a.ndim}" if isinstance(a, np.ndarray) else ""))
    return np.ascontiguousarray(a)  # strided views are copied (stft.rs:21-22 `.to_owned()`)


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def _str(v, name):
    if not isinstance(v, str):
        raise TypeError(f"argument '{name}': expected str")
    return v


def hello_from_bin() -> str:
    """lib.rs:16-19 ("Hello from ssqueeze!"); `version()` identifies the CUDA library."""
    return load().ssq_hello_from_bin().decode()


def version() -> str:
    return load().ssq_version().decode()


def stft(x, n_fft, hop_length, window, padtype):
    """stft.rs:12-19: all five arguments required, positional or keyword.
    Returns (Sx complex128 [n_fft//2+1, n_frames], freqs float64)."""
    x = _f64_1d(x, "x")
    window = _f64_1d(window, "window")
    n_fft, hop = int(n_fft), int(hop_length)
    if n_fft < 0 or hop < 0:
        raise OverflowError("can't convert negative int to unsigned")  # usize extraction
    ctx = default_context()
    lib = load()
    nfq, nfr = C.c_int64(), C.c_int64()
    st = lib.ssq_stft_shape(len(x), n_fft, hop, C.byref(nfq), C.byref(nfr))
    if st != _lib.SSQ_OK:
        raise_status(st, None)
    Sx = np.empty((nfq.value, nfr.value), dtype=np.complex128)
    freqs = np.empty(nfq.value, dtype=np.float64)
    st = lib.ssq_stft_f64(ctx.handle, _ptr(x), len(x), n_fft, hop, _ptr(window), len(window),
                          PAD.get(_str(padtype, "padtype"), 0), _ptr(Sx), _ptr(freqs))
    raise_status(st, ctx.handle)
    return Sx, freqs


def ssq_stft(x, window, n_fft=None, win_len=None, hop_len=1, fs=1.0, padtype="reflect", squeezing="sum",
             gamma=None, *, modulated=False, return_aux=False):
    """ssq_stft.rs:73-85.  Returns (Tx complex128 [n_freqs, n_frames], ssq_freqs).
    `return_aux=True` appends a dict with Sx, dSx (complex128), w (float64) and kb (int32: the destination
    bin of every (source bin, frame), -1 where gated), written by the same kernel that produced Tx."""
    x = _f64_1d(x, "x")
    window = _f64_1d(window, "window")
    n = len(x)
    nf = int(n_fft) if n_fft is not None else min(n, 512)  # ssq_stft.rs:92
    wl = int(win_len) if win_len is not None else len(window)
    hop = int(hop_len)
    if nf < 0 or wl < 0 or hop < 0:
        raise OverflowError("can't convert negative int to unsigned")
    if nf == 0:  # pad = n_fft - 1 underflows (stft_utils.rs:20); also keeps the output shape below in step with the C side
        raise _lib.PanicException("n_fft=0: attempt to subtract with overflow (stft_utils.rs:20)")
    if wl > nf:  # ssq_stft.rs:96-101 (before any shape arithmetic)
        raise ValueError(f"Window length {wl} cannot be greater than n_fft {nf}")
    ctx = default_context()
    lib = load()
    nfq, nfr = C.c_int64(), C.c_int64()
    st = lib.ssq_stft_shape(n, max(nf, 1), hop, C.byref(nfq), C.byref(nfr))
    if st != _lib.SSQ_OK:
        raise_status(st, None)
    shape = (nf // 2 + 1, nfr.value)
    Tx = np.empty(shape, dtype=np.complex128)
    sf = np.empty(shape[0], dtype=np.float64)
    Sx = dSx = w = kb = None
    if return_aux:
        Sx = np.empty(shape, dtype=np.complex128)
        dSx = np.empty(shape, dtype=np.complex128)
        w = np.empty(shape, dtype=np.float64)
        kb = np.empty(shape, dtype=np.int32)
    flags = FLAG_MODULATED if modulated else 0
    g = float(gamma) if gamma is not None else float("nan")  # NaN = not given; negative values never gate
    st = lib.ssq_ssq_stft_f64(ctx.handle, _ptr(x), n, _ptr(window), len(window), nf, wl, hop, float(fs),
                              PAD.get(_str(padtype, "padtype"), 0), SQUEEZE.get(_str(squeezing, "squeezing"), 0),
                              g, flags, _ptr(Tx), _ptr(sf), _ptr(Sx), _ptr(dSx), _ptr(w), _ptr(kb))
    raise_status(st, ctx.handle)
    if return_aux:
        return Tx, sf, dict(Sx=Sx, dSx=dSx, w=w, kb=kb)
    return Tx, sf


def pinned_empty(shape, dtype):
    """A NumPy array in page-locked host memory (ssq_host_alloc; freed with the array): the destination / source that
    lets `ssq_stft_batch` move data at PCIe speed.  Pinning costs ~0.2 s per GB once: keep the array and pass it
    back as `out=`."""
    import weakref
    dt = np.dtype(dtype)
    n = int(np.prod(shape))
    nbytes = max(1, n * dt.itemsize)
    p = C.c_void_p()
    st = load().ssq_host_alloc(C.byref(p), nbytes)
    raise_status(st, None)
    buf = (C.c_char * nbytes).from_address(p.value)
    weakref.finalize(buf, load().ssq_host_free, C.c_void_p(p.value))
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)


def ssq_stft_batch(x, window, n_fft=None, win_len=None, hop_len=1, fs=1.0, padtype="reflect", squeezing="sum",
                   gamma=None, *, modulated=False, out=None, device_out=False):
    """`ssq_stft` (ssq_stft.rs:73-85) for every row of x [channels, n] (float64 or float32) in ONE call -- the
    per-channel Python loop of the reference's multichannel script (tests/stft_ssq_test.py:230-251).
    Returns (Tx complex64 [channels, n_freqs, n_frames], ssq_freqs): the arithmetic of the device is fp32 either way,
    this entry point does not widen the result to complex128 (16 bytes per bin, twice the PCIe time).

    out=None      -> Tx in pinned host memory (`pinned_empty`), written by the chunked H2D | kernel | D2H pipeline of
                     ssq_ssq_stft_host_f32; pass the array back as `out=` to reuse the pinned allocation.
    device_out=True -> Tx is a torch CUDA tensor and never leaves HBM (for a consumer on the device: `extract_ridges`
                     on `ssqueeze_rs_b200.batch.Engine`, a reduction, istft)."""
    if not isinstance(x, np.ndarray) or x.ndim != 2 or x.dtype not in (np.float64, np.float32):
        raise TypeError("argument 'x': expected a 2-D numpy.ndarray [channels, n] of float64 or float32")
    window = _f64_1d(window, "window")
    ch, n = x.shape
    nf = int(n_fft) if n_fft is not None else min(n, 512)
    wl = int(win_len) if win_len is not None else len(window)
    hop = int(hop_len)
    if nf < 0 or wl < 0 or hop < 0:
        raise OverflowError("can't convert negative int to unsigned")
    if nf == 0:
        raise _lib.PanicException("n_fft=0: attempt to subtract with overflow (stft_utils.rs:20)")
    if wl > nf:
        raise ValueError(f"Window length {wl} cannot be greater than n_fft {nf}")
    if wl != len(window):  # the batched C entry points fit the window they are handed
        raise ValueError("ssq_stft_batch: win_len must equal len(window)")
    if ch < 1:
        raise ValueError("x has no channels")
    lib = load()
    nfq, nfr = C.c_int64(), C.c_int64()
    st = lib.ssq_stft_shape(n, max(nf, 1), hop, C.byref(nfq), C.byref(nfr))
    if st != _lib.SSQ_OK:
        raise_status(st, None)
    shape = (ch, nf // 2 + 1, nfr.value)
    sf = np.arange(shape[1], dtype=np.float64) * (float(fs) / 2.0 / max(shape[1] - 1, 1))  # ssq_stft.rs:263-270
    flags = FLAG_MODULATED if modulated else 0
    g = float(gamma) if gamma is not None else float("nan")
    if device_out:
        import torch
        eng = _batch_engine()
        xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(eng.device)
        Tx = eng.ssq_stft(xd, window, nf, hop, float(fs), padtype=_str(padtype, "padtype"),
                          squeezing=_str(squeezing, "squeezing"), gamma=gamma, modulated=modulated)
        return Tx, sf
    x32 = np.ascontiguousarray(x, dtype=np.float32)
    if out is None:
        out = pinned_empty(shape, np.complex64)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.complex64 and out.shape == shape
              and out.flags["C_CONTIGUOUS"]):
        raise ValueError(f"out: expected a C-contiguous complex64 array of shape {shape}")
    ctx = default_context()
    st = lib.ssq_ssq_stft_host_f32(ctx.handle, _ptr(x32), ch, n, _ptr(window), len(window), nf, hop, float(fs),
                                   PAD.get(_str(padtype, "padtype"), 0), SQUEEZE.get(_str(squeezing, "squeezing"), 0),
                                   g, flags, _ptr(out))
    raise_status(st, ctx.handle)
    return out, sf


def stft_batch(x, n_fft, hop_length, window, padtype, *, out=None, device_out=False):
    """`stft` (stft.rs:12-19) for every row of x [channels, n] in one call: (Sx complex64 [channels, n_fft//2+1,
    n_frames], freqs).  `out` / `device_out` as in `ssq_stft_batch`."""
    if not isinstance(x, np.ndarray) or x.ndim != 2 or x.dtype not in (np.float64, np.float32):
        raise TypeError("argument 'x': expected a 2-D numpy.ndarray [channels, n] of float64 or float32")
    window = _f64_1d(window, "window")
    n_fft, hop = int(n_fft), int(hop_length)
    if n_fft < 0 or hop < 0:
        raise OverflowError("can't convert negative int to unsigned")
    ch, n = x.shape
    if ch < 1:
        raise ValueError("x has no channels")
    lib = load()
    nfq, nfr = C.c_int64(), C.c_int64()
    st = lib.ssq_stft_shape(n, n_fft, hop, C.byref(nfq), C.byref(nfr))
    if st != _lib.SSQ_OK:
        raise_status(st, None)
    shape = (ch, nfq.value, nfr.value)
    # Array1::linspace(0.0, 0.5, n_freqs) (stft.rs:40), as the scalar entry point fills it
    freqs = np.arange(nfq.value, dtype=np.float64) * (0.5 / (nfq.value - 1) if nfq.value > 1 else 0.0)
    if nfq.value > 1:
        freqs[-1] = 0.5
    if device_out:
        import torch
        eng = _batch_engine()
        xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(eng.device)
        return eng.stft(xd, window, n_fft, hop, padtype=_str(padtype, "padtype")), freqs
    x32 = np.ascontiguousarray(x, dtype=np.float32)
    if out is None:
        out = pinned_empty(shape, np.complex64)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.complex64 and out.shape == shape
              and out.flags["C_CONTIGUOUS"]):
        raise ValueError(f"out: expected a C-contiguous complex64 array of shape {shape}")
    ctx = default_context()
    st = lib.ssq_stft_host_f32(ctx.handle, _ptr(x32), ch, n, _ptr(window), len(window), n_fft, hop,
                               PAD.get(_str(padtype, "padtype"), 0), _ptr(out))
    raise_status(st, ctx.handle)
    return out, freqs


def ssq_cwt_batch(x, wavelet="gmw", scales=None, fs=None, t=None, ssq_freqs=None, nv=32, padtype="reflect",
                  squeezing="sum", maprange="peak", gamma=None, flipud=True, *, out=None, device_out=False):
    """`ssq_cwt` (ssq_cwt.rs:245-277) for every row of x [channels, n] (float64 or float32) in one call: (Tx complex64
    [channels, n_scales, n], ssq_freqs).  The scalar call returns complex128 -- 9.7 GB per channel at 2^20 samples and
    576 scales; here Tx is complex64, computed in blocks of channels that fit the device and drained into pinned host
    memory (`out=` reuses it), or left on the device as a torch tensor (`device_out=True`, all channels at once)."""
    if not isinstance(x, np.ndarray) or x.ndim != 2 or x.dtype not in (np.float64, np.float32):
        raise TypeError("argument 'x': expected a 2-D numpy.ndarray [channels, n] of float64 or float32")
    ch, n = x.shape
    if ch < 1 or n < 1:
        raise ValueError("x is empty")
    dt = _dt(fs, t)
    sc = _scales(scales, n, nv, False)
    ns = len(sc)
    if ns < 1:
        raise _lib.PanicException("no scales: index out of bounds at ssq_cwt.rs:459")
    import torch
    eng = _batch_engine()
    kw = dict(wavelet=_str(wavelet, "wavelet"), scales=sc, t=np.array([0.0, dt]),  # (dt handed over exactly)
              ssq_freqs=None if ssq_freqs is None else _str(ssq_freqs, "ssq_freqs"), padtype=_str(padtype, "padtype"),
              squeezing=_str(squeezing, "squeezing"), maprange=_str(maprange, "maprange"), gamma=gamma, flipud=flipud)
    x32 = np.ascontiguousarray(x, dtype=np.float32)
    if device_out:
        Tx, sf = eng.ssq_cwt(torch.from_numpy(x32).to(eng.device), return_freqs=True, **kw)
        return Tx, sf
    shape = (ch, ns, n)
    if out is None:
        out = pinned_empty(shape, np.complex64)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.complex64 and out.shape == shape
              and out.flags["C_CONTIGUOUS"]):
        raise ValueError(f"out: expected a C-contiguous complex64 array of shape {shape}")
    per_ch = ns * n * 8
    free, _ = torch.cuda.mem_get_info(eng.device)
    blk = int(max(1, min(ch, (free // 3) // max(per_ch, 1))))  # room for the block's Tx and the FFT workspaces
    sf = None
    stream = torch.cuda.current_stream(eng.device)
    for c0 in range(0, ch, blk):
        c1 = min(ch, c0 + blk)
        Tx, sf = eng.ssq_cwt(torch.from_numpy(x32[c0:c1]).to(eng.device), return_freqs=True, **kw)
        st = load().ssq_memcpy_async(C.c_void_p(out[c0:c1].ctypes.data), C.c_void_p(Tx.data_ptr()), (c1 - c0) * per_ch, 2,
                                     C.c_void_p(stream.cuda_stream if stream.cuda_stream else 1))
        raise_status(st, eng.ctx.handle)
        stream.synchronize()
        del Tx
    return out, sf


_engine = None


def _batch_engine():
    global _engine
    if _engine is None:
        import os
        from .batch import Engine
        _engine = Engine(int(os.environ.get("SSQ_DEVICE", "0")))
    return _engine


def istft(Sx, window, n_fft=None, win_len=None, hop_len=1, N=None, win_exp=1):
    """Inverse of `stft` (Rust framing).  Not in the Rust crate; specified from
    old/ssqueezepy/_stft.py:184-256 with modulated=False and the Rust pad
    offset (n_fft-1)//2."""
    if not isinstance(Sx, np.ndarray) or Sx.ndim != 2 or Sx.dtype != np.complex128:
        raise TypeError("argument 'Sx': expected a 2-D numpy.ndarray of complex128")
    window = _f64_1d(window, "window")
    Sx = np.ascontiguousarray(Sx)
    nfq, nfr = Sx.shape
    nf = int(n_fft) if n_fft else (nfq - 1) * 2
    hop = int(hop_len)
    n_out = int(N) if N else hop * nfr
    if n_out < 1:
        raise ValueError("N must be positive")
    ctx = default_context()
    x = np.empty(n_out, dtype=np.float64)
    st = load().ssq_istft_f64(ctx.handle, _ptr(Sx), nfq, nfr, _ptr(window), len(window), nf, hop, n_out,
                              int(win_exp), _ptr(x))
    raise_status(st, ctx.handle)
    return x


def _bands(cc, cw, n):
    """cc, cw (int arrays [n] or [n, K]) -> contiguous int32 [n, K] each, and K."""
    if (cc is None) != (cw is None):
        raise ValueError("cc and cw go together")
    cc = np.ascontiguousarray(np.asarray(cc).reshape(n, -1), dtype=np.int32)
    cw = np.ascontiguousarray(np.asarray(cw).reshape(n, -1), dtype=np.int32)
    if cc.shape != cw.shape:
        raise ValueError("cc and cw must have the same shape")
    return cc, cw, cc.shape[1]


def issq_stft(Tx, window, n_fft=None, win_len=None, hop_len=1, fs=1.0, *, cc=None, cw=None):
    """Inverse synchrosqueezed STFT (old/ssqueezepy/_ssq_stft.py:139-198).
    Needs hop_len == 1 and a Tx computed with `modulated=True`.  Without `cc` / `cw`: the full inverse, float64
    [n_frames].  With them (int arrays [n_frames] or [n_frames, K] as for `issq_cwt`): the curve bands over the
    frequency rows, [K + 1, n_frames], the last row being the residual."""
    if not isinstance(Tx, np.ndarray) or Tx.ndim != 2 or Tx.dtype != np.complex128:
        raise TypeError("argument 'Tx': expected a 2-D numpy.ndarray of complex128")
    window = _f64_1d(window, "window")
    Tx = np.ascontiguousarray(Tx)
    nfq, nfr = Tx.shape
    nf = int(n_fft) if n_fft else (nfq - 1) * 2
    if cc is not None or cw is not None:
        cc, cw, K = _bands(cc, cw, nfr)
        ctx = default_context()
        y = np.empty((K + 1, nfr), dtype=np.float64)
        st = load().ssq_issq_stft_components_f64(ctx.handle, _ptr(Tx), nfq, nfr, _ptr(window), len(window), nf,
                                                 int(hop_len), float(fs), _ptr(cc), _ptr(cw), K, _ptr(y))
        raise_status(st, ctx.handle)
        return y
    ctx = default_context()
    y = np.empty(nfr, dtype=np.float64)
    st = load().ssq_issq_stft_f64(ctx.handle, _ptr(Tx), nfq, nfr, _ptr(window), len(window), nf, int(hop_len),
                                  float(fs), _ptr(y))
    raise_status(st, ctx.handle)
    return y


def _dt(fs, t):
    # cwt.rs:66-76 / ssq_cwt.rs:283-293
    if t is not None:
        t = _f64_1d(t, "t")
        if len(t) < 2:
            raise ValueError("Time vector must have at least 2 elements")
        return float(t[1] - t[0])
    if fs is not None:
        return 1.0 / float(fs)
    return 1.0


def _scales(scales, n, nv, simd):
    if scales is not None:
        return _f64_1d(scales, "scales").copy()
    lib = load()
    ns = lib.ssq_cwt_default_scales(n, int(nv), int(simd), C.c_void_p(0))
    out = np.empty(max(ns, 0), dtype=np.float64)
    if ns > 0:
        lib.ssq_cwt_default_scales(n, int(nv), int(simd), _ptr(out))
    return out


def _cwt_impl(x, wavelet, scales, fs, t, nv, l1_norm, derivative, padtype, rpadded, simd):
    x = _f64_1d(x, "x")
    n = len(x)
    dt = _dt(fs, t)
    sc = _scales(scales, n, nv, simd)
    ns = len(sc)
    lib = load()
    pl, n1 = C.c_int64(), C.c_int64()
    st = lib.ssq_cwt_shape(n, C.byref(pl), C.byref(n1))
    if st != _lib.SSQ_OK:
        raise_status(st, None)
    cols = pl.value if rpadded else n
    Wx = np.empty((ns, cols), dtype=np.complex128)
    dWx = np.empty((ns, cols), dtype=np.complex128) if derivative else None
    flags = (0 if l1_norm else FLAG_L2_NORM) | (FLAG_RPADDED if rpadded else 0) | (FLAG_SIMD_SCALES if simd else 0)
    ctx = default_context()
    if ns > 0:
        st = lib.ssq_cwt_f64(ctx.handle, _ptr(x), n, 1 if _str(wavelet, "wavelet") == "morlet" else 0, _ptr(sc), ns,
                             dt, PAD.get(_str(padtype, "padtype"), 0), flags, _ptr(Wx), _ptr(dWx))
        raise_status(st, ctx.handle)
    return Wx, sc, dWx


def cwt(x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=True, derivative=False,
        padtype="reflect", rpadded=False, vectorized=True, patience=0):
    """cwt.rs:32-60.  Always a 3-tuple (Wx, scales, dWx | None).  `vectorized`
    selects parallel vs serial code in the reference (same numbers) and
    `patience` is ignored there; both are accepted and ignored here."""
    return _cwt_impl(x, wavelet, scales, fs, t, nv, l1_norm, derivative, padtype, rpadded, simd=False)


def cwt_simd(x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=True, derivative=False,
             padtype="reflect", rpadded=False, vectorized=True, patience=0):
    """cwt_simd.rs:38-66: `cwt` with the exp(p*ln2) default-scale generator."""
    return _cwt_impl(x, wavelet, scales, fs, t, nv, l1_norm, derivative, padtype, rpadded, simd=True)


def ssq_cwt(x, wavelet="gmw", scales=None, fs=None, t=None, ssq_freqs=None, nv=32, padtype="reflect",
            squeezing="sum", maprange="peak", difftype="trig", gamma=None, vectorized=True, flipud=True, *,
            return_aux=False):
    """ssq_cwt.rs:245-277.  Returns (Tx complex128 [n_scales, N], ssq_freqs).
    `difftype` / `vectorized` are ignored as in the reference (:296-297).
    `return_aux=True` (not in the reference) appends a dict with w (float64, the phase transform) and kb (int32: the
    Tx row every (scale, column) was added to, -1: nothing added), written by the reassignment itself."""
    x = _f64_1d(x, "x")
    n = len(x)
    dt = _dt(fs, t)
    sc = _scales(scales, n, nv, False)
    ns = len(sc)
    if ns < 1:
        raise _lib.PanicException("no scales: index out of bounds at ssq_cwt.rs:459")
    dist = 1 if (ssq_freqs is not None and _str(ssq_freqs, "ssq_freqs") == "linear") else 0
    Tx = np.empty((ns, n), dtype=np.complex128)
    sf = np.empty(ns, dtype=np.float64)
    w = np.empty((ns, n), dtype=np.float64) if return_aux else None
    kb = np.empty((ns, n), dtype=np.int32) if return_aux else None
    ctx = default_context()
    g = float(gamma) if gamma is not None else float("nan")
    st = load().ssq_ssq_cwt_f64(ctx.handle, _ptr(x), n, 1 if _str(wavelet, "wavelet") == "morlet" else 0, _ptr(sc),
                                ns, dt, dist, PAD.get(_str(padtype, "padtype"), 0),
                                SQUEEZE.get(_str(squeezing, "squeezing"), 0),
                                1 if _str(maprange, "maprange") == "maximal" else 0, g,
                                0 if flipud else FLAG_NO_FLIPUD, _ptr(Tx), _ptr(sf), _ptr(w), _ptr(kb))
    raise_status(st, ctx.handle)
    if return_aux:
        return Tx, sf, dict(w=w, kb=kb, scales=sc)
    return Tx, sf


def icwt(Wx, wavelet="gmw", scales=None, nv=None, one_int=True, x_len=None, x_mean=0.0, padtype="reflect",
         rpadded=False, l1_norm=True, exact_adm=False):
    """cwt.rs:548-566 (declared in src/ssqueeze/_rs.pyi:62-73, never registered by lib.rs:25-32).
    One-integral reconstruction (default) or the two-integral branch (`one_int=False`, any `x_len <= Wx.shape[1]`:
    row FFTs, Bluestein for lengths that are not powers of two); `nv`, `padtype`, `rpadded` are accepted and unused as
    in the reference.
    `exact_adm=True` (not in the reference) divides by the wavelet's true admissibility integral
    (`adm_ssq`) instead of the placeholders 0.776 / 1.0 of cwt.rs:579-583, so that `icwt(cwt(x))` returns x."""
    if not isinstance(Wx, np.ndarray) or Wx.ndim != 2 or Wx.dtype != np.complex128:
        raise TypeError("argument 'Wx': expected a 2-D numpy.ndarray of complex128")
    if scales is None:
        raise ValueError("Scales must be provided")  # cwt.rs:572-575
    sc = _f64_1d(scales, "scales")
    Wx = np.ascontiguousarray(Wx)
    ns, ncols = Wx.shape
    if len(sc) < ns:
        raise _lib.PanicException("scales shorter than Wx.shape[0]: index out of bounds at cwt.rs:604")
    xl = ncols if x_len is None else int(x_len)
    x = np.empty(max(xl, 0), dtype=np.float64)
    ctx = default_context()
    st = load().ssq_icwt_f64(ctx.handle, _ptr(Wx), ns, ncols, 1 if _str(wavelet, "wavelet") == "morlet" else 0,
                             _ptr(sc), 1 if one_int else 0, xl, float(x_mean),
                             (0 if l1_norm else FLAG_L2_NORM) | (FLAG_ADM_EXACT if exact_adm else 0), _ptr(x))
    raise_status(st, ctx.handle)
    return x


def adm_ssq(wavelet="gmw"):
    """Css = integral psi-hat(w)/w dw of the wavelet `cwt`/`ssq_cwt` evaluate (cwt.rs:492-547); definition
    old/ssqueezepy/utils/cwt_utils.py:28-47."""
    import ctypes
    out = ctypes.c_double(0.0)
    st = load().ssq_cwt_admissibility(1 if _str(wavelet, "wavelet") == "morlet" else 0, ctypes.addressof(out))
    if st != 0:
        raise RuntimeError("ssq_cwt_admissibility failed")
    return out.value


def issq_cwt(Tx, wavelet="gmw", scales=None, cc=None, cw=None):
    """Inversion of `ssq_cwt` (spec old/ssqueezepy/_ssq_cwt.py:313-402; absent from the reference crate):
    x = (2/Css) ln(scales[1]/scales[0]) sum_k Re Tx[k].  `scales` are the ones `ssq_cwt` used; the log-step
    factor is upstream's `const`, which the reference's ssqueeze leaves out of Tx (ssq_cwt.rs:116-222).
    `cc`, `cw` (int arrays [n] or [n, K]: centre row and half-width of K curve bands per column, cc == -1: no
    curve) select the component inversion: returns [K + 1, n], the last row being the residual."""
    if not isinstance(Tx, np.ndarray) or Tx.ndim != 2 or Tx.dtype != np.complex128:
        raise TypeError("argument 'Tx': expected a 2-D numpy.ndarray of complex128")
    if scales is None:
        raise ValueError("Scales must be provided")
    sc = _f64_1d(scales, "scales")
    Tx = np.ascontiguousarray(Tx)
    ns, n = Tx.shape
    ctx = default_context()
    wid = 1 if _str(wavelet, "wavelet") == "morlet" else 0
    if cc is not None or cw is not None:
        cc, cw, K = _bands(cc, cw, n)
        x = np.empty((K + 1, n), dtype=np.float64)
        st = load().ssq_issq_cwt_components_f64(ctx.handle, _ptr(Tx), ns, n, wid, _ptr(sc), _ptr(cc), _ptr(cw), K,
                                                _ptr(x))
        raise_status(st, ctx.handle)
        return x
    x = np.empty(n, dtype=np.float64)
    st = load().ssq_issq_cwt_f64(ctx.handle, _ptr(Tx), ns, n, wid, _ptr(sc), _ptr(x))
    raise_status(st, ctx.handle)
    return x


def extract_ridges(Tf, scales, penalty=2.0, n_ridges=1, bw=15, transform="cwt", get_params=False, parallel=True, *,
                   return_E=False):
    """Forward/backward penalised ridge tracking on a time-frequency map (SURVEY 8f rank 4).  The reference crate
    declares `ridge::extraction` and leaves it empty (rust/src/ridge/{mod,extraction}.rs); signature, semantics and
    return values are upstream's `extract_ridges` (old/ssqueezepy/ridge_extraction.py:11-150): ridge_idxs int
    [n_time, n_ridges] (and ridge_f, ridge_e with `get_params`).  Tf: complex128 (float64 arithmetic, eps = EPS64) or
    complex64 (float32, EPS32) [n_freq, n_time]; `parallel` is accepted and ignored (the result is that of upstream's
    sequential code).  `return_E=True` appends the diagnostic E = -log(energy / max + eps) of every ridge."""
    if not isinstance(Tf, np.ndarray) or Tf.ndim != 2 or Tf.dtype not in (np.complex128, np.complex64):
        raise TypeError("argument 'Tf': expected a 2-D numpy.ndarray of complex128 or complex64")
    Tf = np.ascontiguousarray(Tf)
    is64 = Tf.dtype == np.complex128
    rdt = np.float64 if is64 else np.float32
    sc = np.ascontiguousarray(np.asarray(scales, dtype=np.float64).reshape(-1))
    nf, nt = Tf.shape
    if len(sc) != nf:
        raise ValueError(f"scales has {len(sc)} entries, Tf has {nf} rows")
    tr = 0 if _str(transform, "transform") == "cwt" else 1
    idx = np.empty((nt, int(n_ridges)), dtype=np.int32)
    rf = np.empty((nt, int(n_ridges)), dtype=rdt) if get_params else None
    re_ = np.empty((nt, int(n_ridges)), dtype=rdt) if get_params else None
    E = np.empty((int(n_ridges), nf, nt), dtype=rdt) if return_E else None
    ctx = default_context()
    st = load().ssq_extract_ridges_host(ctx.handle, _ptr(Tf), 1 if is64 else 0, nf, nt, _ptr(sc), float(penalty),
                                        int(n_ridges), int(bw), tr, _ptr(idx), _ptr(rf), _ptr(re_), _ptr(E))
    raise_status(st, ctx.handle)
    out = (idx.astype(int), rf, re_) if get_params else idx.astype(int)
    if return_E:
        return (out + (E,)) if get_params else (out, E)
    return out


# ---- wavelet generators (src/ssqueeze/_rs.pyi:91-132; rust/src/wavelets/{morlet,gmw}.rs) ----------------------
def _wavelet_call(fn, kind, w, n, *args):
    out = np.empty(n, dtype=np.complex128)
    st = fn(kind, _ptr(w) if w is not None else C.c_void_p(0), n, *args, _ptr(out))
    raise_status(st, None)
    return out


def morlet(w, mu=6.0, dtype="float64"):
    """morlet.rs:59-76.  psi-hat(w) complex128; `dtype` is accepted and unused as in the reference."""
    w = _f64_1d(w, "w")
    return _wavelet_call(load().ssq_wavelet_morlet, 0, w, len(w), 1.0, float(mu))


def morlet_freq(n=1024, scale=1.0, mu=6.0, dtype="float64"):
    """morlet.rs:79-101: psi-hat on xifn(scale, n)."""
    return _wavelet_call(load().ssq_wavelet_morlet, 1, None, int(n), float(scale), float(mu))


def morlet_time(n=1024, scale=1.0, mu=6.0, dtype="float64"):
    """morlet.rs:104-145: the time-domain wavelet."""
    return _wavelet_call(load().ssq_wavelet_morlet, 2, None, int(n), float(scale), float(mu))


def gmw(w, gamma=3.0, beta=60.0, norm="bandpass", order=0, dtype="float64"):
    """gmw.rs:226-258 (ValueError for gamma <= 0, beta < 0, order < 0)."""
    w = _f64_1d(w, "w")
    return _wavelet_call(load().ssq_wavelet_gmw, 0, w, len(w), 1.0, float(gamma), float(beta),
                         1 if _str(norm, "norm").lower() == "bandpass" else 0, int(order))


def gmw_freq(n=1024, scale=1.0, gamma=3.0, beta=60.0, norm="bandpass", order=0, dtype="float64"):
    """gmw.rs:261-281."""
    return _wavelet_call(load().ssq_wavelet_gmw, 1, None, int(n), float(scale), float(gamma), float(beta),
                         1 if _str(norm, "norm").lower() == "bandpass" else 0, int(order))


def gmw_time(n=1024, scale=1.0, gamma=3.0, beta=60.0, norm="bandpass", order=0, dtype="float64"):
    """gmw.rs:284-327."""
    return _wavelet_call(load().ssq_wavelet_gmw, 2, None, int(n), float(scale), float(gamma), float(beta),
                         1 if _str(norm, "norm").lower() == "bandpass" else 0, int(order))


def gmw_center_frequency(gamma=3.0, beta=60.0, kind="peak"):
    """gmw.rs:331-357: "peak" | "energy", anything else raises ValueError."""
    k = {"peak": 0, "energy": 1}.get(_str(kind, "kind"), 2)
    out = C.c_double(0.0)
    st = load().ssq_wavelet_gmw_center_frequency(float(gamma), float(beta), k, C.byref(out))
    if st == _lib.SSQ_EINVAL:
        raise ValueError(f"Unknown center frequency kind: {kind}")
    raise_status(st, None)
    return out.value

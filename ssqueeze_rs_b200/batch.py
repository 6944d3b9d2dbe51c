"""Multichannel throughput path: replaces the per-channel Python loop around
`_rs.ssq_stft` (tests/stft_ssq_test.py:230-251 of the reference) by batched
C-ABI calls on device buffers, and shards channel blocks across the GPUs of one
box (channels are independent; no collective, host gather only).

`Engine` wraps one device context.  Pointer-level methods take raw device/host
addresses (what the C ABI takes); tensor-level helpers accept torch CUDA
tensors (torch is used for device memory and streams only).
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib
from ._lib import PAD, SQUEEZE, Context, load, raise_status


def _wptr(window):
    w = np.ascontiguousarray(window, dtype=np.float64)
    return w, C.c_void_p(w.ctypes.data)


def _bands(cc, cw, ch, n, device):
    """cc, cw of the component inversions -> contiguous int32 CUDA tensors [ch, n, K] and K.  cc: int32 CUDA tensor
    [ch, n, K] (what `Engine.extract_ridges` returns) or [ch, n] (one band); cw: a tensor of the same shape, or an int
    broadcast to it.  Raises ValueError before anything is launched."""
    import numbers

    import torch
    if cc is None or cw is None:
        raise ValueError("cc and cw go together")
    if not (isinstance(cc, torch.Tensor) and cc.dtype == torch.int32 and cc.device == device):
        raise ValueError(f"cc must be an int32 tensor on {device}")
    if cc.dim() == 2:
        cc = cc.unsqueeze(-1)
    if cc.dim() != 3 or tuple(cc.shape[:2]) != (ch, n):
        raise ValueError(f"cc has shape {tuple(cc.shape)}; expected [{ch}, {n}, K] or [{ch}, {n}]")
    if isinstance(cw, numbers.Integral) and not isinstance(cw, bool):
        if not -2**31 <= int(cw) < 2**31:
            raise ValueError("cw does not fit int32")
        cw = torch.full_like(cc, int(cw))
    elif isinstance(cw, torch.Tensor) and cw.dtype == torch.int32 and cw.device == device:
        if cw.dim() == 2:
            cw = cw.unsqueeze(-1)
        if cw.shape != cc.shape:
            raise ValueError(f"cw has shape {tuple(cw.shape)}, cc {tuple(cc.shape)}")
    else:
        raise ValueError(f"cw must be an int or an int32 tensor on {device}")
    return cc.contiguous(), cw.contiguous(), cc.shape[2]


class Engine:
    def __init__(self, device: int = 0):
        self.ctx = Context(device)
        self.device = device

    def last_kernel_name(self) -> str:
        return self.ctx.last_kernel_name()

    # ---- pointer level ---------------------------------------------------
    def ssq_stft_ptr(self, d_x, channels, n, window, n_fft, hop, fs, d_Tx, padtype="reflect", squeezing="sum",
                     gamma=None, modulated=False, x_stride=0, diag=None):
        """diag: optional (d_Sx, d_dSx, d_w, d_kb) device addresses (0 = not wanted) -> the diagnostic twin."""
        w, wp = _wptr(window)
        args = (self.ctx.handle, C.c_void_p(d_x), channels, n, x_stride or n, wp, len(w),
                int(n_fft), int(hop), float(fs), PAD.get(padtype, 0),
                SQUEEZE.get(squeezing, 0), float("nan") if gamma is None else float(gamma),
                _lib.FLAG_MODULATED if modulated else 0, C.c_void_p(d_Tx))
        if diag is None:
            st = load().ssq_ssq_stft_batch_f32(*args)
        else:
            st = load().ssq_ssq_stft_batch_diag_f32(*args, *[C.c_void_p(a or 0) for a in diag])
        raise_status(st, self.ctx.handle)

    def stft_ptr(self, d_x, channels, n, window, n_fft, hop, d_Sx, padtype="reflect", x_stride=0):
        w, wp = _wptr(window)
        st = load().ssq_stft_batch_f32(self.ctx.handle, C.c_void_p(d_x), channels, n, x_stride or n, wp, len(w),
                                       int(n_fft), int(hop), PAD.get(padtype, 0), C.c_void_p(d_Sx))
        raise_status(st, self.ctx.handle)

    def istft_ptr(self, d_Sx, channels, n_freqs, n_frames, window, n_fft, hop, n_out, d_x, win_exp=1):
        w, wp = _wptr(window)
        st = load().ssq_istft_batch_f32(self.ctx.handle, C.c_void_p(d_Sx), channels, n_freqs, n_frames, wp, len(w),
                                        int(n_fft), int(hop), int(n_out), int(win_exp), C.c_void_p(d_x))
        raise_status(st, self.ctx.handle)

    def issq_stft_ptr(self, d_Tx, channels, n_freqs, n_frames, window, n_fft, fs, d_y):
        w, wp = _wptr(window)
        st = load().ssq_issq_stft_batch_f32(self.ctx.handle, C.c_void_p(d_Tx), channels, n_freqs, n_frames, wp,
                                            len(w), int(n_fft), float(fs), C.c_void_p(d_y))
        raise_status(st, self.ctx.handle)

    def ssq_stft_host(self, h_x, channels, n, window, n_fft, hop, fs, h_Tx, padtype="reflect", squeezing="sum",
                      gamma=None, modulated=False):
        """Host (pinned) buffers in/out; copies inside the call (synchronous)."""
        w, wp = _wptr(window)
        st = load().ssq_ssq_stft_host_f32(self.ctx.handle, C.c_void_p(h_x), channels, n, wp, len(w), int(n_fft),
                                          int(hop), float(fs), PAD.get(padtype, 0), SQUEEZE.get(squeezing, 0),
                                          float("nan") if gamma is None else float(gamma),
                                          _lib.FLAG_MODULATED if modulated else 0, C.c_void_p(h_Tx))
        raise_status(st, self.ctx.handle)

    # ---- tensor level (torch CUDA tensors) ----------------------------------
    def _bind_stream(self):
        import torch
        h = torch.cuda.current_stream(self.device).cuda_stream
        # handle 0 is the legacy default stream; the C ABI reserves NULL for "the context's own
        # stream", so name the legacy stream explicitly (cudaStreamLegacy == 0x1)
        self.ctx.set_stream(h if h else 1)

    def ssq_stft(self, x, window, n_fft=512, hop_len=32, fs=1.0, out=None, return_aux=False, **kw):
        """x: float32 CUDA tensor [channels, n] -> complex64 [channels, n_freqs, n_frames].
        return_aux: also a dict of device tensors Sx, dSx (complex64), w (float32), kb (int32) written by the same
        kernel (diagnostic variant; parity tests)."""
        import torch
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        ch, n = x.shape
        nfq, nfr = n_fft // 2 + 1, (n - 1) // hop_len + 1
        if out is None:
            out = torch.empty((ch, nfq, nfr), dtype=torch.complex64, device=x.device)
        self._bind_stream()
        if not return_aux:
            self.ssq_stft_ptr(x.data_ptr(), ch, n, window, n_fft, hop_len, fs, out.data_ptr(), x_stride=x.stride(0), **kw)
            return out
        aux = dict(Sx=torch.empty_like(out), dSx=torch.empty_like(out),
                   w=torch.empty((ch, nfq, nfr), dtype=torch.float32, device=x.device),
                   kb=torch.empty((ch, nfq, nfr), dtype=torch.int32, device=x.device))
        self.ssq_stft_ptr(x.data_ptr(), ch, n, window, n_fft, hop_len, fs, out.data_ptr(), x_stride=x.stride(0),
                          diag=(aux["Sx"].data_ptr(), aux["dSx"].data_ptr(), aux["w"].data_ptr(), aux["kb"].data_ptr()),
                          **kw)
        return out, aux

    def stft(self, x, window, n_fft, hop_len, out=None, padtype="reflect"):
        import torch
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        ch, n = x.shape
        nfq, nfr = n_fft // 2 + 1, (n - 1) // hop_len + 1
        if out is None:
            out = torch.empty((ch, nfq, nfr), dtype=torch.complex64, device=x.device)
        self._bind_stream()
        self.stft_ptr(x.data_ptr(), ch, n, window, n_fft, hop_len, out.data_ptr(), padtype, x_stride=x.stride(0))
        return out

    def istft(self, Sx, window, n_fft, hop_len, N=None, win_exp=1, out=None):
        import torch
        assert Sx.is_cuda and Sx.dtype == torch.complex64 and Sx.dim() == 3 and Sx.is_contiguous()
        ch, nfq, nfr = Sx.shape
        n_out = N or hop_len * nfr
        if out is None:
            out = torch.empty((ch, n_out), dtype=torch.float32, device=Sx.device)
        assert out.shape == (ch, n_out) and out.dtype == torch.float32 and out.is_contiguous()
        self._bind_stream()
        self.istft_ptr(Sx.data_ptr(), ch, nfq, nfr, window, n_fft, hop_len, n_out, out.data_ptr(), win_exp)
        return out

    def issq_stft(self, Tx, window, n_fft, fs=1.0, cc=None, cw=None):
        """Tx: complex64 CUDA [channels, n_freqs, n_frames] (hop 1, modulated) -> y float32 [channels, n_frames].
        With `cc`, `cw` (see `issq_cwt`): the curve bands over the frequency rows, float32 [channels, K + 1, n_frames],
        row K the residual."""
        import torch
        assert Tx.is_cuda and Tx.dtype == torch.complex64 and Tx.dim() == 3 and Tx.is_contiguous()
        ch, nfq, nfr = Tx.shape
        if cc is not None or cw is not None:
            cc, cw, K = _bands(cc, cw, ch, nfr, Tx.device)
            y = torch.empty((ch, K + 1, nfr), dtype=torch.float32, device=Tx.device)
            w, wp = _wptr(window)
            self._bind_stream()
            st = load().ssq_issq_stft_components_batch_f32(self.ctx.handle, C.c_void_p(Tx.data_ptr()), ch, nfq, nfr, wp,
                                                           len(w), int(n_fft), float(fs), C.c_void_p(cc.data_ptr()),
                                                           C.c_void_p(cw.data_ptr()), K, C.c_void_p(y.data_ptr()))
            raise_status(st, self.ctx.handle)
            return y
        out = torch.empty((ch, nfr), dtype=torch.float32, device=Tx.device)
        self._bind_stream()
        self.issq_stft_ptr(Tx.data_ptr(), ch, nfq, nfr, window, n_fft, fs, out.data_ptr())
        return out


    # ---- CWT family --------------------------------------------------------------
    def _cwt_args(self, x, scales, fs, t, nv, simd=False):
        import torch
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        ch, n = x.shape
        if scales is None:
            ns = load().ssq_cwt_default_scales(n, int(nv), int(simd), C.c_void_p(0))
            sc = np.empty(ns, dtype=np.float64)
            load().ssq_cwt_default_scales(n, int(nv), int(simd), C.c_void_p(sc.ctypes.data))
        else:
            sc = np.ascontiguousarray(scales, dtype=np.float64)
        dt = float(t[1] - t[0]) if t is not None else (1.0 / float(fs) if fs is not None else 1.0)
        return ch, n, sc, dt

    def cwt(self, x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=True, derivative=False,
            padtype="reflect", rpadded=False, simd=False):
        """x: float32 CUDA [channels, n] -> Wx complex64 [channels, ns, n|pad_len] (and dWx)."""
        import torch
        ch, n, sc, dt = self._cwt_args(x, scales, fs, t, nv, simd)
        pl = C.c_int64()
        load().ssq_cwt_shape(n, C.byref(pl), None)
        cols = pl.value if rpadded else n
        Wx = torch.empty((ch, len(sc), cols), dtype=torch.complex64, device=x.device)
        dWx = torch.empty_like(Wx) if derivative else None
        flags = (0 if l1_norm else _lib.FLAG_L2_NORM) | (_lib.FLAG_RPADDED if rpadded else 0)
        self._bind_stream()
        st = load().ssq_cwt_batch_f32(self.ctx.handle, C.c_void_p(x.data_ptr()), ch, n, x.stride(0),
                                      1 if wavelet == "morlet" else 0, C.c_void_p(sc.ctypes.data), len(sc), dt,
                                      PAD.get(padtype, 0), flags, C.c_void_p(Wx.data_ptr()),
                                      C.c_void_p(dWx.data_ptr() if derivative else 0))
        raise_status(st, self.ctx.handle)
        return (Wx, dWx) if derivative else Wx

    def ssq_cwt(self, x, wavelet="gmw", scales=None, fs=None, t=None, ssq_freqs=None, nv=32, padtype="reflect",
                squeezing="sum", maprange="peak", gamma=None, flipud=True, out=None, return_freqs=False,
                return_aux=False):
        """x: float32 CUDA [channels, n] -> Tx complex64 [channels, ns, n].
        return_aux: (Tx, ssq_freqs, dict(w float32, kb int32, scales)) -- diagnostics written by the reassignment."""
        import torch
        ch, n, sc, dt = self._cwt_args(x, scales, fs, t, nv)
        if out is None:
            out = torch.empty((ch, len(sc), n), dtype=torch.complex64, device=x.device)
        sf = np.empty(len(sc), dtype=np.float64)
        self._bind_stream()
        args = (self.ctx.handle, C.c_void_p(x.data_ptr()), ch, n, x.stride(0),
                1 if wavelet == "morlet" else 0, C.c_void_p(sc.ctypes.data), len(sc), dt,
                1 if ssq_freqs == "linear" else 0, PAD.get(padtype, 0),
                SQUEEZE.get(squeezing, 0), 1 if maprange == "maximal" else 0,
                float("nan") if gamma is None else float(gamma),
                0 if flipud else _lib.FLAG_NO_FLIPUD, C.c_void_p(out.data_ptr()), C.c_void_p(sf.ctypes.data))
        if return_aux:
            w = torch.empty((ch, len(sc), n), dtype=torch.float32, device=x.device)
            kb = torch.empty((ch, len(sc), n), dtype=torch.int32, device=x.device)
            st = load().ssq_ssq_cwt_batch_diag_f32(*args, C.c_void_p(w.data_ptr()), C.c_void_p(kb.data_ptr()))
            raise_status(st, self.ctx.handle)
            return out, sf, dict(w=w, kb=kb, scales=sc)
        st = load().ssq_ssq_cwt_batch_f32(*args)
        raise_status(st, self.ctx.handle)
        return (out, sf) if return_freqs else out


    def icwt(self, Wx, scales, wavelet="gmw", l1_norm=True, x_mean=0.0, exact_adm=False, x_len=None):
        """Wx: complex64 CUDA [channels, ns, n_cols] -> x float32 [channels, x_len] (one-integral branch)."""
        import torch
        assert Wx.is_cuda and Wx.dtype == torch.complex64 and Wx.dim() == 3 and Wx.is_contiguous()
        ch, ns, ncols = Wx.shape
        sc = np.ascontiguousarray(scales, dtype=np.float64)
        xl = ncols if x_len is None else int(x_len)
        x = torch.empty((ch, xl), dtype=torch.float32, device=Wx.device)
        flags = (0 if l1_norm else _lib.FLAG_L2_NORM) | (_lib.FLAG_ADM_EXACT if exact_adm else 0)
        self._bind_stream()
        st = load().ssq_icwt_batch_f32(self.ctx.handle, C.c_void_p(Wx.data_ptr()), ch, ns, ncols,
                                       1 if wavelet == "morlet" else 0, C.c_void_p(sc.ctypes.data), 1, xl,
                                       float(x_mean), flags, C.c_void_p(x.data_ptr()))
        raise_status(st, self.ctx.handle)
        return x

    def issq_cwt(self, Tx, scales, wavelet="gmw", cc=None, cw=None):
        """Tx: complex64 CUDA [channels, ns, n] -> x float32 [channels, n] (full inversion).
        With `cc`, `cw`: the component inversion (old/ssqueezepy/_ssq_cwt.py:380-402) of K curve bands, float32
        [channels, K + 1, n], row K the residual.  cc: int32 CUDA tensor [channels, n, K] of centre rows, e.g. the
        indices `extract_ridges` returns (cc == -1: no curve at that column), or [channels, n] for one band; cw: the
        half-widths, a tensor of the same shape or an int.  Band c of column j is the rows clip(cc - cw, 0, ns) ..
        clip(cc + cw, 0, ns), clipped on the device; 1 <= K <= 16."""
        import torch
        assert Tx.is_cuda and Tx.dtype == torch.complex64 and Tx.dim() == 3 and Tx.is_contiguous()
        ch, ns, n = Tx.shape
        sc = np.ascontiguousarray(scales, dtype=np.float64)
        if cc is not None or cw is not None:
            cc, cw, K = _bands(cc, cw, ch, n, Tx.device)
            x = torch.empty((ch, K + 1, n), dtype=torch.float32, device=Tx.device)
            self._bind_stream()
            st = load().ssq_issq_cwt_components_batch_f32(self.ctx.handle, C.c_void_p(Tx.data_ptr()), ch, ns, n,
                                                          1 if wavelet == "morlet" else 0, C.c_void_p(sc.ctypes.data),
                                                          C.c_void_p(cc.data_ptr()), C.c_void_p(cw.data_ptr()), K,
                                                          C.c_void_p(x.data_ptr()))
            raise_status(st, self.ctx.handle)
            return x
        x = torch.empty((ch, n), dtype=torch.float32, device=Tx.device)
        self._bind_stream()
        st = load().ssq_issq_cwt_batch_f32(self.ctx.handle, C.c_void_p(Tx.data_ptr()), ch, ns, n,
                                           1 if wavelet == "morlet" else 0, C.c_void_p(sc.ctypes.data),
                                           C.c_void_p(x.data_ptr()))
        raise_status(st, self.ctx.handle)
        return x

    def extract_ridges(self, Tf, scales, penalty=2.0, n_ridges=1, bw=15, transform="cwt", get_params=False):
        """Tf: complex64 CUDA [channels, n_freq, n_time] (e.g. the Tx `ssq_stft` / `ssq_cwt` just wrote) -> ridge indices
        int32 [channels, n_time, n_ridges] (and ridge_f, ridge_e float32 with get_params).  The map never leaves HBM."""
        import torch
        assert Tf.is_cuda and Tf.dim() == 3 and Tf.is_contiguous() and Tf.dtype in (torch.complex64, torch.complex128)
        ch, nf, nt = Tf.shape
        is64 = Tf.dtype == torch.complex128
        sc = np.ascontiguousarray(np.asarray(scales, dtype=np.float64).reshape(-1))
        assert len(sc) == nf
        idx = torch.empty((ch, nt, n_ridges), dtype=torch.int32, device=Tf.device)
        rdt = torch.float64 if is64 else torch.float32
        rf = torch.empty((ch, nt, n_ridges), dtype=rdt, device=Tf.device) if get_params else None
        re_ = torch.empty((ch, nt, n_ridges), dtype=rdt, device=Tf.device) if get_params else None
        self._bind_stream()
        st = load().ssq_extract_ridges_batch(self.ctx.handle, C.c_void_p(Tf.data_ptr()), 1 if is64 else 0, ch, nf, nt,
                                             C.c_void_p(sc.ctypes.data), float(penalty), int(n_ridges), int(bw),
                                             0 if transform == "cwt" else 1, C.c_void_p(idx.data_ptr()),
                                             C.c_void_p(rf.data_ptr() if get_params else 0),
                                             C.c_void_p(re_.data_ptr() if get_params else 0), C.c_void_p(0))
        raise_status(st, self.ctx.handle)
        return (idx, rf, re_) if get_params else idx

    def default_scales(self, n, nv=32, simd=False):
        ns = load().ssq_cwt_default_scales(int(n), int(nv), int(simd), C.c_void_p(0))
        sc = np.empty(ns, dtype=np.float64)
        load().ssq_cwt_default_scales(int(n), int(nv), int(simd), C.c_void_p(sc.ctypes.data))
        return sc


class SsqStftStream:
    """Streaming ssq_stft over chunks of an interleaved [samples, channels] recording (int16 or
    float32 CUDA tensors): the B200 replacement of the dask `map_overlap` caller
    (tests/stft_ssq_test.py:218-283 of the reference).  `push(chunk)` returns the frames that
    became complete, complex64 [channels, n_freqs, frames]; concatenated along frames they equal
    `Engine.ssq_stft` on the whole recording (no re-padding at chunk seams).  Each output can be handed,
    masked or not, straight to `IstftStream.push` (transform="stft" for istft; modulated=True, hop 1 for
    issq_stft)."""

    def __init__(self, engine: "Engine", channels, n_total, max_chunk, window, n_fft=512, hop_len=32, fs=1.0,
                 padtype="reflect", squeezing="sum", gamma=None, transform="ssq_stft", modulated=False):
        """transform: "ssq_stft" (frames of Tx) or "stft" (frames of Sx: the caller of tests/stft_test.py:215-271)."""
        if transform not in ("ssq_stft", "stft"):
            raise ValueError("transform must be 'ssq_stft' or 'stft'")
        self.eng = engine
        self.channels, self.n_freqs, self.max_chunk = int(channels), int(n_fft) // 2 + 1, int(max_chunk)
        w, wp = _wptr(window)
        h = C.c_void_p()
        st = load().ssq_stream_create_ex(engine.ctx.handle, int(channels), int(n_total), int(max_chunk), wp, len(w),
                                         int(n_fft), int(hop_len), float(fs), PAD.get(padtype, 0),
                                         SQUEEZE.get(squeezing, 0), float("nan") if gamma is None else float(gamma),
                                         1 if transform == "stft" else 0, _lib.FLAG_MODULATED if modulated else 0,
                                         C.byref(h))
        raise_status(st, engine.ctx.handle)
        self._h = h

    @property
    def total_frames(self) -> int:
        return int(load().ssq_stream_total_frames(self._h))

    def push(self, chunk, scale=1.0):
        import torch
        assert chunk.is_cuda and chunk.dim() == 2 and chunk.shape[1] == self.channels and chunk.is_contiguous()
        n_new = chunk.shape[0]
        frames = int(load().ssq_stream_frames_after(self._h, n_new))
        out = torch.empty((self.channels, self.n_freqs, max(frames, 0)), dtype=torch.complex64, device=chunk.device)
        self.eng._bind_stream()
        fw = C.c_int64()
        fn = {torch.int16: load().ssq_stream_push_i16, torch.float32: load().ssq_stream_push_f32}[chunk.dtype]
        st = fn(self._h, C.c_void_p(chunk.data_ptr()), n_new, float(scale),
                C.c_void_p(out.data_ptr() if frames > 0 else 0), C.byref(fw))
        raise_status(st, self.eng.ctx.handle)
        assert fw.value == max(frames, 0)
        return out

    def close(self):
        if self._h:
            load().ssq_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CwtStream:
    """Streaming cwt / ssq_cwt over chunks of an interleaved [samples, channels] recording (int16 or float32 CUDA
    tensors): the dask `map_overlap(depth=overlap, boundary="reflect")` caller of the reference's CWT scripts
    (tests/cwt_test.py:117-119,187-193 of the reference), DESIGN §3.6b.  Block b covers output columns
    [b block, (b + 1) block) and is the reference's call on its extended input x~[b block - overlap, (b + 1) block +
    overlap) (x~: the recording mirrored with the edge sample repeated at both ends), trimmed to its own columns.
    `push(chunk)` returns the columns of the blocks that became complete, complex64 [channels, ns, cols]; the result
    does not depend on how the recording is cut into pushes.  The CWT has no seam-exact stream: a block differs from
    the whole-signal transform near its seams by an amount that falls with overlap / scale (DESIGN §3.6b).

        cs = CwtStream(eng, 384, n, max_chunk=1 << 18, block=1 << 17, overlap=1 << 14, fs=30000.0)
        for Tx in RecordingFeeder(eng, rec, None, chunk=1 << 18, scale=0.195, stream=cs):
            power += Tx.abs().square().sum(dim=2)   # [384, ns]: the reduction stays on the device

    The arguments are those of `Engine.ssq_cwt` (transform="ssq_cwt") and `Engine.cwt` (transform="cwt", l1_norm).
    scales default to `Engine.default_scales(block + 2 overlap, nv)`, what the reference's call on a full block uses."""

    def __init__(self, engine: "Engine", channels, n_total, max_chunk, block, overlap, wavelet="gmw", scales=None,
                 fs=None, t=None, nv=32, transform="ssq_cwt", padtype="reflect", squeezing="sum", maprange="peak",
                 ssq_freqs="log", gamma=None, flipud=True, l1_norm=True):
        if transform not in ("ssq_cwt", "cwt"):
            raise ValueError("transform must be 'ssq_cwt' or 'cwt'")
        self.eng, self.transform = engine, transform
        self.channels, self.max_chunk = int(channels), int(max_chunk)
        if scales is None:
            sc = engine.default_scales(int(block) + 2 * int(overlap), nv) if int(block) >= 1 else np.ones(1)
        else:
            sc = scales
        self.scales = np.ascontiguousarray(sc, dtype=np.float64)
        self.ns = len(self.scales)
        dt = float(t[1] - t[0]) if t is not None else (1.0 / float(fs) if fs is not None else 1.0)
        if transform == "cwt":
            mode, flags = 2, (0 if l1_norm else _lib.FLAG_L2_NORM)
        else:
            mode, flags = 3, (0 if flipud else _lib.FLAG_NO_FLIPUD)
        h = C.c_void_p()
        st = load().ssq_stream_create_cwt(engine.ctx.handle, self.channels, int(n_total), self.max_chunk, int(block),
                                          int(overlap), mode, 1 if wavelet == "morlet" else 0,
                                          C.c_void_p(self.scales.ctypes.data), self.ns, dt,
                                          1 if ssq_freqs == "linear" else 0, PAD.get(padtype, 0),
                                          SQUEEZE.get(squeezing, 0), 1 if maprange == "maximal" else 0,
                                          float("nan") if gamma is None else float(gamma), flags, C.byref(h))
        raise_status(st, engine.ctx.handle)
        self._h = h

    @property
    def total_frames(self) -> int:
        """Output columns over the whole recording: n_total."""
        return int(load().ssq_stream_total_frames(self._h))

    def ssq_freqs(self, last=False):
        """The ssq grid (float64 [ns]) of the full blocks, or of the last block (its own under maprange="maximal")."""
        f = np.empty(self.ns, dtype=np.float64)
        raise_status(load().ssq_stream_ssq_freqs(self._h, 1 if last else 0, C.c_void_p(f.ctypes.data)),
                     self.eng.ctx.handle)
        return f

    def push(self, chunk, scale=1.0):
        import torch
        assert chunk.is_cuda and chunk.dim() == 2 and chunk.shape[1] == self.channels and chunk.is_contiguous()
        n_new = chunk.shape[0]
        cols = max(int(load().ssq_stream_frames_after(self._h, n_new)), 0)
        out = torch.empty((self.channels, self.ns, cols), dtype=torch.complex64, device=chunk.device)
        self.eng._bind_stream()
        fw = C.c_int64()
        fn = {torch.int16: load().ssq_stream_push_i16, torch.float32: load().ssq_stream_push_f32}[chunk.dtype]
        st = fn(self._h, C.c_void_p(chunk.data_ptr()), n_new, float(scale),
                C.c_void_p(out.data_ptr() if cols > 0 else 0), C.byref(fw))
        raise_status(st, self.eng.ctx.handle)
        assert fw.value == cols
        return out

    def close(self):
        if getattr(self, "_h", None):
            load().ssq_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class IstftStream:
    """Streaming inverse over chunks of frames (ssq_istream_*, DESIGN §3.4c): `push(Sx_chunk)` takes the next frames,
    complex64 CUDA [channels, n_freqs, frames] as `SsqStftStream` / `RecordingFeeder` yield them, and returns the
    output samples that became final.  Concatenated over pushes they are `Engine.istft(Sx, window, n_fft, hop_len, N,
    win_exp)` (transform="istft") or `Engine.issq_stft(Tx, window, n_fft, fs)` (transform="issq_stft", hop_len 1) of
    the whole Sx / Tx, without ever holding it:

        inv = IstftStream(eng, 384, n_frames, (chunk + 512) // 32 + 2, win, 512, 32, N=n,  # frames of one feeder chunk
                          out="i16_interleaved", scale=0.195)
        for Sx in RecordingFeeder(eng, rec, win, 512, 32, chunk=chunk, scale=0.195, transform="stft"):
            y = inv.push(mask * Sx)      # int16 [samples, 384], the counts of the filtered recording

    out: "f32" -> float32 [channels, samples], "f32_interleaved" -> float32 [samples, channels], "i16_interleaved" ->
    int16 [samples, channels] (round to nearest even, saturated).  Samples are multiplied by float32(1 / scale)."""

    _FORMATS = {"f32": 0, "f32_interleaved": 1, "i16_interleaved": 2}
    _TRANSFORMS = {"istft": 0, "issq_stft": 1}

    def __init__(self, engine: "Engine", channels, n_frames_total, max_frames, window, n_fft=512, hop_len=32, N=None,
                 win_exp=1, transform="istft", fs=1.0, out="f32", scale=1.0):
        if transform not in self._TRANSFORMS:
            raise ValueError("transform must be 'istft' or 'issq_stft'")
        if out not in self._FORMATS:
            raise ValueError("out must be 'f32', 'f32_interleaved' or 'i16_interleaved'")
        self.eng, self.out, self.scale = engine, out, float(scale)
        self.channels, self.n_freqs = int(channels), int(n_fft) // 2 + 1
        w, wp = _wptr(window)
        h = C.c_void_p()
        st = load().ssq_istream_create(engine.ctx.handle, int(channels), int(n_frames_total), int(N or 0),
                                       int(max_frames), wp, len(w), int(n_fft), int(hop_len), int(win_exp),
                                       self._TRANSFORMS[transform], float(fs), self._FORMATS[out], C.byref(h))
        raise_status(st, engine.ctx.handle)
        self._h = h

    @property
    def total_samples(self) -> int:
        return int(load().ssq_istream_total_samples(self._h))

    def push(self, Sx_chunk):
        import torch
        assert Sx_chunk.is_cuda and Sx_chunk.dtype == torch.complex64 and Sx_chunk.dim() == 3
        assert Sx_chunk.shape[:2] == (self.channels, self.n_freqs) and Sx_chunk.is_contiguous()
        n_new = Sx_chunk.shape[2]
        k = max(int(load().ssq_istream_samples_after(self._h, n_new)), 0)
        shape = (self.channels, k) if self.out == "f32" else (k, self.channels)
        dtype = torch.int16 if self.out == "i16_interleaved" else torch.float32
        y = torch.empty(shape, dtype=dtype, device=Sx_chunk.device)
        self.eng._bind_stream()
        sw = C.c_int64()
        st = load().ssq_istream_push(self._h, C.c_void_p(Sx_chunk.data_ptr()), n_new, self.scale,
                                     C.c_void_p(y.data_ptr() if k > 0 else 0), C.byref(sw))
        raise_status(st, self.eng.ctx.handle)
        assert sw.value == k
        return y

    def close(self):
        if getattr(self, "_h", None):
            load().ssq_istream_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ParquetRecording:
    """A (samples, channels) recording stored as parquet columns -- the on-disk format of the reference's real-data
    scripts (tests/stft_test.py:374-377 read the whole table into memory with pq.read_table(...).to_pandas().values
    and hand it to dask in chunks of 10^6 samples).  This wrapper reads it batch by batch instead: it has the `shape`,
    `dtype` and forward slicing `rec[a:b]` that `RecordingFeeder` needs, and returns C-contiguous float32 (or int16)
    [b - a, channels] blocks; memory stays at one batch.  Slices must advance monotonically (a stream)."""

    ndim = 2

    def __init__(self, path, columns=None, batch_rows=1 << 16):
        import pyarrow.parquet as pq
        self._pf = pq.ParquetFile(str(path), memory_map=True)
        names = [f.name for f in self._pf.schema_arrow]
        self.columns = list(columns) if columns is not None else names
        missing = [c for c in self.columns if c not in names]
        if missing:
            raise ValueError(f"columns not in the file: {missing}")
        import pyarrow as pa
        types = [self._pf.schema_arrow.field(c).type for c in self.columns]
        self.dtype = np.dtype(np.int16) if all(pa.types.is_int16(t) for t in types) else np.dtype(np.float32)
        self.shape = (int(self._pf.metadata.num_rows), len(self.columns))
        self._batch_rows = int(batch_rows)
        self._it = None
        self._buf = np.empty((0, self.shape[1]), dtype=self.dtype)
        self._buf_start = 0  # global row of _buf[0]

    def _more(self):
        if self._it is None:
            self._it = self._pf.iter_batches(batch_size=self._batch_rows, columns=self.columns)
        b = next(self._it)
        blk = np.empty((b.num_rows, self.shape[1]), dtype=self.dtype)
        for j, c in enumerate(self.columns):  # column-major on disk -> interleaved rows
            blk[:, j] = b.column(b.schema.get_field_index(c)).to_numpy(zero_copy_only=False)
        return blk

    def __getitem__(self, key):
        if not isinstance(key, slice) or key.step not in (None, 1):
            raise TypeError("ParquetRecording supports forward slices rec[a:b] only")
        a, b, _ = key.indices(self.shape[0])
        if a < self._buf_start:
            raise ValueError("ParquetRecording is a stream: slices must not go backwards")
        while self._buf_start + len(self._buf) < b:
            drop = min(max(a - self._buf_start, 0), len(self._buf))
            self._buf = np.concatenate([self._buf[drop:], self._more()], axis=0)
            self._buf_start += drop
        lo = a - self._buf_start
        return np.ascontiguousarray(self._buf[lo:lo + (b - a)])


class RecordingFeeder:
    """Host half of the streaming path: walks an interleaved (samples, channels) recording that lies in HOST memory --
    a NumPy array or a memory-mapped int16 / float32 file, as the reference's multichannel scripts open them
    (tests/stft_ssq_test.py:218-283, tests/stft_test.py:374-377) -- in chunks, through the library's ring of pinned
    staging buffers (ssq_feeder_*: host copy | H2D | transform overlap), and yields the frames of every chunk as they
    become complete: complex64 CUDA tensors [channels, n_freqs, frames] that stay on the device for a consumer
    (ridge extraction, band power, a reduction).  Concatenated along frames they equal `Engine.ssq_stft` on the whole
    recording bit for bit.

        rec = np.memmap("probe.dat", dtype=np.int16, mode="r").reshape(-1, 384)
        with RecordingFeeder(eng, rec, np.hanning(512), scale=0.195, fs=30000.0) as feed:
            for Tx in feed:              # [384, 257, frames of this chunk]
                ...

    With transform="stft" the chunks are frames of Sx, and `IstftStream` turns them back into samples chunk by chunk
    (filter in the time-frequency plane, then write the result out):

        for Sx in RecordingFeeder(eng, rec, win, 512, 32, chunk=1 << 18, scale=0.195, transform="stft"):
            y = inv.push(mask * Sx)      # inv = IstftStream(..., out="i16_interleaved", scale=0.195)

    stream: a `CwtStream` or `SsqStftStream` made for this recording's channels and length; the feeder drives it
    (chunks of at most its max_chunk) and yields its outputs, [channels, ns or n_freqs, columns]; window and the
    transform arguments are then unused.  The caller keeps the stream and closes it.
    """

    def __init__(self, engine: "Engine", recording, window, n_fft=512, hop_len=32, fs=1.0, chunk=1 << 16, scale=1.0,
                 padtype="reflect", squeezing="sum", gamma=None, depth=3, transform="ssq_stft", modulated=False,
                 stream=None):
        rec = recording
        if rec.ndim != 2:
            raise ValueError("recording must be [samples, channels]")
        if rec.dtype not in (np.int16, np.float32):
            raise ValueError("recording dtype must be int16 or float32")
        self.eng, self.rec, self.scale = engine, rec, float(scale)
        self.n_total, self.channels = int(rec.shape[0]), int(rec.shape[1])
        self.chunk = int(min(max(1, chunk), self.n_total))
        self._own_stream = stream is None
        if stream is None:
            self.stream = SsqStftStream(engine, self.channels, self.n_total, self.chunk, window, n_fft, hop_len, fs,
                                        padtype=padtype, squeezing=squeezing, gamma=gamma, transform=transform,
                                        modulated=modulated)
        else:
            if stream.channels != self.channels:
                raise ValueError(f"stream has {stream.channels} channels, the recording {self.channels}")
            self.stream = stream
            self.chunk = min(self.chunk, stream.max_chunk)
        self.rows = self.stream.ns if isinstance(self.stream, CwtStream) else self.stream.n_freqs
        h = C.c_void_p()
        st = load().ssq_feeder_create(self.stream._h, 0 if rec.dtype == np.int16 else 1, int(depth), C.byref(h))
        raise_status(st, engine.ctx.handle)
        self._h = h
        self.pos = 0

    @property
    def total_frames(self) -> int:
        return self.stream.total_frames

    def push_next(self):
        """Queues the next chunk; returns the CUDA tensor of its frames (None at the end of the recording)."""
        import torch
        if self.pos >= self.n_total:
            return None
        n_new = min(self.chunk, self.n_total - self.pos)
        src = self.rec[self.pos:self.pos + n_new]
        if not src.flags["C_CONTIGUOUS"]:
            src = np.ascontiguousarray(src)
        frames = max(int(load().ssq_stream_frames_after(self.stream._h, n_new)), 0)
        # (torch's caching allocator hands the same blocks back once the consumer drops the previous chunks)
        out = torch.empty((self.channels, self.rows, frames), dtype=torch.complex64, device=self.eng.device)
        self.eng._bind_stream()
        fw = C.c_int64()
        st = load().ssq_feeder_push(self._h, C.c_void_p(src.ctypes.data), n_new, self.scale,
                                    C.c_void_p(out.data_ptr() if frames > 0 else 0), C.byref(fw))
        raise_status(st, self.eng.ctx.handle)
        assert fw.value == frames
        self.pos += n_new
        return out

    def __iter__(self):
        while True:
            out = self.push_next()
            if out is None:
                return
            yield out

    def close(self):
        if getattr(self, "_h", None):
            load().ssq_feeder_destroy(self._h)
            self._h = None
        if getattr(self, "stream", None) and getattr(self, "_own_stream", True):
            self.stream.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shard_channels(channels: int, n_devices: int):
    """Contiguous channel blocks: device g gets [g*C/G, (g+1)*C/G) (SURVEY 8e)."""
    return [(g * channels // n_devices, (g + 1) * channels // n_devices) for g in range(n_devices)]


class ChannelSharder:
    """One host thread + one context per device; numpy host arrays in/out.
    No inter-GPU traffic: each device works on its own channel block and writes
    its block of the host result (host gather only)."""

    def __init__(self, devices):
        self.devices = list(devices)
        self.engines = [Engine(d) for d in self.devices]

    def ssq_stft(self, x: np.ndarray, window, n_fft=512, hop_len=32, fs=1.0, **kw) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        ch, n = x.shape
        nfq, nfr = n_fft // 2 + 1, (n - 1) // hop_len + 1
        out = np.empty((ch, nfq, nfr), dtype=np.complex64)
        errs = []

        def work(eng, lo, hi):
            try:
                if hi > lo:
                    eng.ssq_stft_host(x[lo:hi].ctypes.data, hi - lo, n, window, n_fft, hop_len, fs,
                                      out[lo:hi].ctypes.data, **kw)
            except BaseException as e:  # surfaced below
                errs.append(e)

        ths = [threading.Thread(target=work, args=(e, lo, hi))
               for e, (lo, hi) in zip(self.engines, shard_channels(ch, len(self.engines)))]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]
        return out

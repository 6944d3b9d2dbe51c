"""ctypes binding of libssqcuda.so (include/ssqcuda.h).  Fails loudly when the
library is missing -- there is no Python/NumPy fallback on the product path."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libssqcuda.so"


def lib_path() -> str:
    return os.environ.get("SSQCUDA_LIB", os.path.join(_HERE, _LIB_NAME))


class SsqError(RuntimeError):
    """CUDA / allocation / unsupported-configuration failure."""


class PanicException(BaseException):
    """Mirror of pyo3_runtime.PanicException (derives from BaseException): raised
    for inputs on which the reference Rust code panics (hop 0, empty x, window
    shorter than n_fft in `stft`, ...)."""


SSQ_OK, SSQ_EINVAL, SSQ_ECUDA, SSQ_ENOMEM, SSQ_EUNSUPPORTED, SSQ_EPANIC = range(6)

PAD = {"reflect": 0, "zero": 1}
SQUEEZE = {"sum": 0, "lebesgue": 1}
FLAG_MODULATED, FLAG_NO_FLIPUD, FLAG_L2_NORM, FLAG_RPADDED, FLAG_SIMD_SCALES, FLAG_ADM_EXACT = 1, 2, 4, 8, 16, 32

c_i64, c_int, c_dbl, c_u32, c_vp = C.c_int64, C.c_int, C.c_double, C.c_uint, C.c_void_p
P_dbl = C.POINTER(C.c_double)

# name -> (restype, argtypes); every symbol include/ssqcuda.h declares
SIGNATURES = {
    "ssq_version": (C.c_char_p, []),
    "ssq_hello_from_bin": (C.c_char_p, []),
    "ssq_device_count": (c_int, []),
    "ssq_ctx_create": (c_int, [c_int, C.POINTER(c_vp)]),
    "ssq_ctx_destroy": (None, [c_vp]),
    "ssq_last_error": (C.c_char_p, [c_vp]),
    "ssq_ctx_set_stream": (c_int, [c_vp, c_vp]),
    "ssq_ctx_synchronize": (c_int, [c_vp]),
    "ssq_ctx_set_option": (c_int, [c_vp, C.c_char_p, c_i64]),
    "ssq_ctx_launch_count": (C.c_uint64, [c_vp]),
    "ssq_ctx_last_kernel_ms": (C.c_float, [c_vp]),
    "ssq_ctx_last_kernel_name": (C.c_char_p, [c_vp]),
    "ssq_stft_shape": (c_int, [c_i64, c_int, c_int, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "ssq_cwt_shape": (c_int, [c_i64, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "ssq_cwt_default_scales": (c_i64, [c_i64, c_int, c_int, c_vp]),
    "ssq_stft_f64": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_i64, c_int, c_vp, c_vp]),
    "ssq_ssq_stft_f64": (c_int, [c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_dbl, c_int, c_int,
                                 c_dbl, c_u32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "ssq_istft_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_i64, c_int, c_vp]),
    "ssq_issq_stft_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_vp]),
    "ssq_cwt_f64": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_i64, c_dbl, c_int, c_u32, c_vp, c_vp]),
    "ssq_ssq_cwt_f64": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_i64, c_dbl, c_int, c_int, c_int, c_int,
                                c_dbl, c_u32, c_vp, c_vp, c_vp, c_vp]),
    "ssq_ssq_cwt_batch_diag_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_dbl, c_int, c_int,
                                           c_int, c_int, c_dbl, c_u32, c_vp, c_vp, c_vp, c_vp]),
    "ssq_icwt_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_int, c_i64, c_dbl, c_u32, c_vp]),
    "ssq_cwt_admissibility": (c_int, [c_int, c_vp]),
    "ssq_issq_cwt_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp]),
    "ssq_issq_cwt_components_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_int, c_vp]),
    "ssq_issq_cwt_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp]),
    "ssq_issq_cwt_components_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_int,
                                                  c_vp]),
    "ssq_issq_stft_components_f64": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_vp, c_vp,
                                             c_int, c_vp]),
    "ssq_issq_stft_components_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_dbl, c_vp,
                                                   c_vp, c_int, c_vp]),
    "ssq_icwt_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_int, c_i64, c_dbl, c_u32, c_vp]),
    "ssq_ssq_stft_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl,
                                       c_int, c_int, c_dbl, c_u32, c_vp]),
    "ssq_ssq_stft_batch_diag_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl,
                                            c_int, c_int, c_dbl, c_u32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "ssq_stft_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "ssq_istft_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_i64, c_int,
                                    c_vp]),
    "ssq_issq_stft_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_dbl, c_vp]),
    "ssq_cwt_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_dbl, c_int, c_u32,
                                  c_vp, c_vp]),
    "ssq_ssq_cwt_batch_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_dbl, c_int, c_int,
                                      c_int, c_int, c_dbl, c_u32, c_vp, c_vp]),
    "ssq_stft_host_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "ssq_ssq_stft_host_f32": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_int, c_int,
                                      c_dbl, c_u32, c_vp]),
    "ssq_wavelet_morlet": (c_int, [c_int, c_vp, c_i64, c_dbl, c_dbl, c_vp]),
    "ssq_wavelet_gmw": (c_int, [c_int, c_vp, c_i64, c_dbl, c_dbl, c_dbl, c_int, c_int, c_vp]),
    "ssq_wavelet_gmw_center_frequency": (c_int, [c_dbl, c_dbl, c_int, C.POINTER(c_dbl)]),
    "ssq_extract_ridges_batch": (c_int, [c_vp, c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_dbl, c_int, c_int, c_int, c_vp,
                                         c_vp, c_vp, c_vp]),
    "ssq_extract_ridges_host": (c_int, [c_vp, c_vp, c_int, c_i64, c_i64, c_vp, c_dbl, c_int, c_int, c_int, c_vp, c_vp,
                                        c_vp, c_vp]),
    "ssq_stream_create": (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_int, c_int, c_dbl,
                                  C.POINTER(c_vp)]),
    "ssq_stream_create_ex": (c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_int, c_int, c_dbl,
                                     c_int, C.c_uint, C.POINTER(c_vp)]),
    "ssq_stream_destroy": (None, [c_vp]),
    "ssq_stream_total_frames": (c_i64, [c_vp]),
    "ssq_stream_frames_after": (c_i64, [c_vp, c_i64]),
    "ssq_stream_push_i16": (c_int, [c_vp, c_vp, c_i64, C.c_float, c_vp, C.POINTER(c_i64)]),
    "ssq_stream_push_f32": (c_int, [c_vp, c_vp, c_i64, C.c_float, c_vp, C.POINTER(c_i64)]),
    "ssq_stream_create_cwt": (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, c_int, c_int, c_vp, c_i64, c_dbl,
                                      c_int, c_int, c_int, c_int, c_dbl, C.c_uint, C.POINTER(c_vp)]),
    "ssq_stream_ssq_freqs": (c_int, [c_vp, c_int, c_vp]),
    "ssq_feeder_create": (c_int, [c_vp, c_int, c_int, C.POINTER(c_vp)]),
    "ssq_feeder_destroy": (None, [c_vp]),
    "ssq_feeder_push": (c_int, [c_vp, c_vp, c_i64, C.c_float, c_vp, C.POINTER(c_i64)]),
    "ssq_istream_create": (c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int, c_dbl,
                                   c_int, C.POINTER(c_vp)]),
    "ssq_istream_destroy": (None, [c_vp]),
    "ssq_istream_total_samples": (c_i64, [c_vp]),
    "ssq_istream_samples_after": (c_i64, [c_vp, c_i64]),
    "ssq_istream_push": (c_int, [c_vp, c_vp, c_i64, C.c_float, c_vp, C.POINTER(c_i64)]),
    "ssq_host_alloc": (c_int, [C.POINTER(c_vp), C.c_size_t]),
    "ssq_host_free": (None, [c_vp]),
    "ssq_memcpy_async": (c_int, [c_vp, c_vp, C.c_size_t, c_int, c_vp]),
    "ssq_device_numa_node": (c_int, [c_int, C.POINTER(c_int)]),
    "ssq_host_alloc_near": (c_int, [C.POINTER(c_vp), C.c_size_t, c_int]),
}

_lib = None
_lib_lock = threading.Lock()


def load():
    """Load libssqcuda.so once; ImportError (loud) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.path.exists(path) and "SSQCUDA_LIB" not in os.environ:
            # a fresh checkout (the .so is not tracked): compile it in-tree once if nvcc is around;
            # this is a build step, not a fallback -- without the library every call still fails
            try:
                import importlib.util
                spec = importlib.util.spec_from_file_location(
                    "__graft_entry__", os.path.join(os.path.dirname(_HERE), "__graft_entry__.py"))
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                mod.build_cuda()
            except Exception:
                pass
        if not os.path.exists(path):
            raise ImportError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the build is stale
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def raise_status(st: int, ctx):
    if st == SSQ_OK:
        return
    msg = load().ssq_last_error(ctx)
    msg = msg.decode("utf-8", "replace") if msg else f"status {st}"
    if st == SSQ_EINVAL:
        raise ValueError(msg)
    if st == SSQ_EPANIC:
        raise PanicException(msg)
    if st == SSQ_ENOMEM:
        raise MemoryError(msg)
    raise SsqError(msg)


class Context:
    """One device context (stream, workspaces, table cache).  Not thread-safe."""

    def __init__(self, device: int = 0):
        lib = load()
        h = c_vp()
        st = lib.ssq_ctx_create(int(device), C.byref(h))
        if st != SSQ_OK:
            raise_status(st, None)
        self._h = h
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def set_stream(self, cuda_stream_ptr):
        raise_status(load().ssq_ctx_set_stream(self._h, c_vp(cuda_stream_ptr or 0)), self._h)

    def set_option(self, name: str, value: int):
        """Context option (include/ssqcuda.h ssq_ctx_set_option): ``no_h32r``, ``no_r1024``, ``no_r256`` and
        ``no_cwt_fused`` select the reference paths of the cross-checks, ``upstream_framing`` the upstream framing.
        An unknown name raises ValueError."""
        raise_status(load().ssq_ctx_set_option(self._h, name.encode(), int(value)), self._h)

    def synchronize(self):
        raise_status(load().ssq_ctx_synchronize(self._h), self._h)

    def launch_count(self) -> int:
        return int(load().ssq_ctx_launch_count(self._h))

    def last_kernel_ms(self) -> float:
        return float(load().ssq_ctx_last_kernel_ms(self._h))

    def last_kernel_name(self) -> str:
        return load().ssq_ctx_last_kernel_name(self._h).decode()

    def close(self):
        if self._h:
            load().ssq_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_tls = threading.local()


def default_context() -> Context:
    """Per-thread default context on device $SSQ_DEVICE (default 0), mirroring the
    reference's re-entrant, state-free functions."""
    dev = int(os.environ.get("SSQ_DEVICE", "0"))
    ctxs = getattr(_tls, "ctxs", None)
    if ctxs is None:
        ctxs = _tls.ctxs = {}
    if dev not in ctxs:
        ctxs[dev] = Context(dev)
    return ctxs[dev]

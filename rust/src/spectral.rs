// spectral.rs -- the #[pyfunction]s of rust/src/spectral/{stft,ssq_stft,cwt,cwt_simd,ssq_cwt}.rs with everything that
// ran inside `Python::allow_threads` replaced by ONE call into libssqcuda (arithmetic: fp32 on the B200; the arrays
// that cross this boundary keep the reference's dtypes, float64 / complex128).  Argument parsing, defaults, the
// PyValueErrors and the return arity are the reference's.  Python mirror of this file (what the tests drive, since
// the build image has no Rust toolchain): ssqueeze_rs_b200/_rs.py.
use ndarray::{Array1, Array2};
use num_complex::Complex64;
use numpy::{AllowTypeChange, IntoPyArray, PyArrayLikeDyn, PyReadonlyArray1, PyReadonlyArray2};
use pyo3::exceptions::PyValueError;
use pyo3::prelude::*;
use std::os::raw::c_int;

use crate::ffi;

fn pad_code(padtype: &str) -> c_int {
    if padtype == "zero" { 1 } else { 0 } // anything else: reflect (stft.rs:25-29, ssq_stft.rs:124-128, cwt.rs:88-92)
}
fn squeeze_code(s: &str) -> c_int {
    if s == "lebesgue" { 1 } else { 0 } // anything else: sum (ssq_stft.rs:292-296, ssq_cwt.rs:199-206)
}
fn wavelet_code(w: &str) -> c_int {
    if w == "morlet" { 1 } else { 0 } // anything else is GMW(3, 60) (cwt.rs:496-541)
}

/// stft.rs:12-95
#[pyfunction]
pub fn stft<'py>(
    py: Python<'py>,
    x: PyReadonlyArray1<f64>,
    n_fft: usize,
    hop_length: usize,
    window: PyReadonlyArray1<f64>,
    padtype: &str,
) -> PyResult<(PyObject, PyObject)> {
    let x_s = x.as_array().to_owned();
    let w_s = window.as_array().to_owned();
    let (mut nfq, mut nfr) = (0i64, 0i64);
    // n_frames = (n - 1) / hop + 1, n_freqs = n_fft / 2 + 1 (stft.rs:32-34); hop 0 / empty x: the reference panics
    let st = unsafe { ffi::ssq_stft_shape(x_s.len() as i64, n_fft as c_int, hop_length as c_int, &mut nfq, &mut nfr) };
    ffi::check(st, std::ptr::null())?;
    let mut sx = Array2::<Complex64>::zeros((nfq as usize, nfr as usize));
    let mut freqs = Array1::<f64>::zeros(nfq as usize);
    let pad = pad_code(padtype);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_stft_f64(c, x_s.as_ptr(), x_s.len() as i64, n_fft as c_int, hop_length as c_int, w_s.as_ptr(),
                              w_s.len() as i64, pad, sx.as_mut_ptr() as *mut f64, freqs.as_mut_ptr())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok((sx.into_pyarray(py).into_py(py), freqs.into_pyarray(py).into_py(py)))
}

/// ssq_stft.rs:73-313
#[pyfunction]
#[pyo3(signature = (x, window, n_fft=None, win_len=None, hop_len=1, fs=1.0, padtype="reflect", squeezing="sum", gamma=None, modulated=false))]
pub fn ssq_stft<'py>(
    py: Python<'py>,
    x: PyReadonlyArray1<f64>,
    window: PyReadonlyArray1<f64>,
    n_fft: Option<usize>,
    win_len: Option<usize>,
    hop_len: usize,
    fs: f64,
    padtype: &str,
    squeezing: &str,
    gamma: Option<f64>,
    modulated: bool,
) -> PyResult<(PyObject, PyObject)> {
    let x_s = x.as_array().to_owned();
    let w_s = window.as_array().to_owned();
    let n = x_s.len();
    let n_fft = n_fft.unwrap_or(n.min(512)); // :92
    let win_len = win_len.unwrap_or(w_s.len()); // :93
    if win_len > n_fft {
        return Err(PyValueError::new_err(format!("Window length {} cannot be greater than n_fft {}", win_len, n_fft))); // :96-101
    }
    let n_freqs = n_fft / 2 + 1;
    let n_frames = (n + n_fft - 1 - n_fft) / hop_len + 1; // :182-183 (panics for n = 0 / hop_len = 0 like the reference)
    let mut tx = Array2::<Complex64>::zeros((n_freqs, n_frames));
    let mut ssq_freqs = Array1::<f64>::zeros(n_freqs);
    let (pad, sq) = (pad_code(padtype), squeeze_code(squeezing));
    let flags = if modulated { ffi::SSQ_FLAG_MODULATED } else { 0 };
    let g = gamma.unwrap_or(f64::NAN); // NaN = not given -> 10 eps (:258-261); a negative value never gates (:23)
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_ssq_stft_f64(c, x_s.as_ptr(), n as i64, w_s.as_ptr(), w_s.len() as i64, n_fft as c_int,
                                  win_len as c_int, hop_len as c_int, fs, pad, sq, g, flags,
                                  tx.as_mut_ptr() as *mut f64, ssq_freqs.as_mut_ptr(), std::ptr::null_mut(),
                                  std::ptr::null_mut(), std::ptr::null_mut(), std::ptr::null_mut())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok((tx.into_pyarray(py).into_py(py), ssq_freqs.into_pyarray(py).into_py(py)))
}

/// `ssq_stft` for every row of x [channels, n] in one call (the per-channel Python loop of
/// tests/stft_ssq_test.py:230-251): complex64 out -- the device computes in fp32 either way, widening to complex128
/// would double the PCIe time.  Host pipeline H2D | kernel | D2H inside ssq_ssq_stft_host_f32.
#[pyfunction]
#[pyo3(signature = (x, window, n_fft=None, hop_len=1, fs=1.0, padtype="reflect", squeezing="sum", gamma=None, modulated=false))]
pub fn ssq_stft_batch<'py>(
    py: Python<'py>,
    x: PyReadonlyArray2<f64>,
    window: PyReadonlyArray1<f64>,
    n_fft: Option<usize>,
    hop_len: usize,
    fs: f64,
    padtype: &str,
    squeezing: &str,
    gamma: Option<f64>,
    modulated: bool,
) -> PyResult<(PyObject, PyObject)> {
    let xa = x.as_array();
    let (channels, n) = (xa.shape()[0], xa.shape()[1]);
    let x32: Vec<f32> = xa.iter().map(|v| *v as f32).collect(); // row-major [channels, n]
    let w_s = window.as_array().to_owned();
    let n_fft = n_fft.unwrap_or(n.min(512));
    if w_s.len() > n_fft {
        return Err(PyValueError::new_err(format!("Window length {} cannot be greater than n_fft {}", w_s.len(), n_fft)));
    }
    let n_freqs = n_fft / 2 + 1;
    let n_frames = (n - 1) / hop_len + 1;
    let mut tx = ndarray::Array3::<num_complex::Complex32>::zeros((channels, n_freqs, n_frames));
    let (pad, sq) = (pad_code(padtype), squeeze_code(squeezing));
    let flags = if modulated { ffi::SSQ_FLAG_MODULATED } else { 0 };
    let g = gamma.unwrap_or(f64::NAN);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_ssq_stft_host_f32(c, x32.as_ptr(), channels as i64, n as i64, w_s.as_ptr(), w_s.len() as i64,
                                       n_fft as c_int, hop_len as c_int, fs, pad, sq, g, flags,
                                       tx.as_mut_ptr() as *mut f32)
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    let ssq_freqs = Array1::<f64>::from_shape_fn(n_freqs, |i| (i as f64) * 0.5 * fs / ((n_freqs as f64) - 1.0)); // :42-54
    Ok((tx.into_pyarray(py).into_py(py), ssq_freqs.into_pyarray(py).into_py(py)))
}

/// `stft` for every row of x [channels, n] in one call (ssq_stft_host_f32); complex64 out.
#[pyfunction]
pub fn stft_batch<'py>(
    py: Python<'py>,
    x: PyReadonlyArray2<f64>,
    n_fft: usize,
    hop_length: usize,
    window: PyReadonlyArray1<f64>,
    padtype: &str,
) -> PyResult<(PyObject, PyObject)> {
    let xa = x.as_array();
    let (channels, n) = (xa.shape()[0], xa.shape()[1]);
    let x32: Vec<f32> = xa.iter().map(|v| *v as f32).collect();
    let w_s = window.as_array().to_owned();
    let (mut nfq, mut nfr) = (0i64, 0i64);
    let st = unsafe { ffi::ssq_stft_shape(n as i64, n_fft as c_int, hop_length as c_int, &mut nfq, &mut nfr) };
    ffi::check(st, std::ptr::null())?;
    let mut sx = ndarray::Array3::<num_complex::Complex32>::zeros((channels, nfq as usize, nfr as usize));
    let pad = pad_code(padtype);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_stft_host_f32(c, x32.as_ptr(), channels as i64, n as i64, w_s.as_ptr(), w_s.len() as i64,
                                   n_fft as c_int, hop_length as c_int, pad, sx.as_mut_ptr() as *mut f32)
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    let freqs = Array1::<f64>::linspace(0.0, 0.5, nfq as usize); // stft.rs:40
    Ok((sx.into_pyarray(py).into_py(py), freqs.into_pyarray(py).into_py(py)))
}

/// Inverse of `stft` (north star; spec old/ssqueezepy/_stft.py:184-256 in the crate's framing)
#[pyfunction]
#[pyo3(signature = (sx, window, n_fft=None, win_len=None, hop_len=1, n=None, win_exp=1))]
pub fn istft<'py>(
    py: Python<'py>,
    sx: PyReadonlyArray2<Complex64>,
    window: PyReadonlyArray1<f64>,
    n_fft: Option<usize>,
    win_len: Option<usize>,
    hop_len: usize,
    n: Option<usize>,
    win_exp: i32,
) -> PyResult<PyObject> {
    let _ = win_len;
    let s = sx.as_array().as_standard_layout().to_owned();
    let w_s = window.as_array().to_owned();
    let (nfq, nfr) = (s.shape()[0], s.shape()[1]);
    let n_fft = n_fft.unwrap_or((nfq - 1) * 2);
    let n_out = n.unwrap_or(hop_len * nfr);
    let mut out = Array1::<f64>::zeros(n_out);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_istft_f64(c, s.as_ptr() as *const f64, nfq as i64, nfr as i64, w_s.as_ptr(), w_s.len() as i64,
                               n_fft as c_int, hop_len as c_int, n_out as i64, win_exp, out.as_mut_ptr())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok(out.into_pyarray(py).into_py(py))
}

type Bands<'py> = Option<PyArrayLikeDyn<'py, i32, AllowTypeChange>>;

/// cc / cw of the component inversions (old/ssqueezepy/_ssq_cwt.py:380-402): int arrays [n] (one band) or [n, K], each
/// read as int32 [n][K]; None when neither is given.  Errors are raised before any device work.
fn bands(cc: Bands<'_>, cw: Bands<'_>, n: usize) -> PyResult<Option<(Vec<i32>, Vec<i32>, usize)>> {
    let (cc, cw) = match (cc, cw) {
        (None, None) => return Ok(None),
        (Some(cc), Some(cw)) => (cc, cw),
        _ => return Err(PyValueError::new_err("cc and cw go together")),
    };
    let (a, b) = (cc.as_array(), cw.as_array());
    if n == 0 || a.len() % n != 0 || b.len() % n != 0 {
        return Err(PyValueError::new_err(format!("cannot reshape cc / cw of {} / {} elements to [{n}, K]", a.len(), b.len())));
    }
    if a.len() != b.len() {
        return Err(PyValueError::new_err("cc and cw must have the same shape"));
    }
    let k = a.len() / n;
    Ok(Some((a.iter().copied().collect(), b.iter().copied().collect(), k)))
}

/// Inverse synchrosqueezed STFT (old/ssqueezepy/_ssq_stft.py:139-198; hop_len must be 1, Tx from modulated=True).
/// With `cc`, `cw`: the curve bands over the frequency rows, [K + 1, n_frames], the residual last.
#[pyfunction]
#[pyo3(signature = (tx, window, n_fft=None, win_len=None, hop_len=1, fs=1.0, *, cc=None, cw=None))]
#[allow(clippy::too_many_arguments)]
pub fn issq_stft<'py>(
    py: Python<'py>,
    tx: PyReadonlyArray2<Complex64>,
    window: PyReadonlyArray1<f64>,
    n_fft: Option<usize>,
    win_len: Option<usize>,
    hop_len: usize,
    fs: f64,
    cc: Bands<'py>,
    cw: Bands<'py>,
) -> PyResult<PyObject> {
    let _ = win_len;
    let t = tx.as_array().as_standard_layout().to_owned();
    let w_s = window.as_array().to_owned();
    let (nfq, nfr) = (t.shape()[0], t.shape()[1]);
    let n_fft = n_fft.unwrap_or((nfq - 1) * 2);
    if let Some((cc, cw, k)) = bands(cc, cw, nfr)? {
        let mut y = Array2::<f64>::zeros((k + 1, nfr));
        let st = py.allow_threads(|| {
            ffi::with_ctx(|c| unsafe {
                ffi::ssq_issq_stft_components_f64(c, t.as_ptr() as *const f64, nfq as i64, nfr as i64, w_s.as_ptr(),
                                                  w_s.len() as i64, n_fft as c_int, hop_len as c_int, fs, cc.as_ptr(),
                                                  cw.as_ptr(), k as c_int, y.as_mut_ptr())
            })
        });
        ffi::with_ctx(|c| ffi::check(st, c))?;
        return Ok(y.into_pyarray(py).into_py(py));
    }
    let mut y = Array1::<f64>::zeros(nfr);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_issq_stft_f64(c, t.as_ptr() as *const f64, nfq as i64, nfr as i64, w_s.as_ptr(), w_s.len() as i64,
                                   n_fft as c_int, hop_len as c_int, fs, y.as_mut_ptr())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok(y.into_pyarray(py).into_py(py))
}

fn dt_of(fs: Option<f64>, t: &Option<PyReadonlyArray1<f64>>) -> PyResult<f64> {
    // cwt.rs:66-76 / ssq_cwt.rs:283-293
    if let Some(t) = t {
        let t = t.as_array();
        if t.len() < 2 {
            return Err(PyValueError::new_err("Time vector must have at least 2 elements"));
        }
        return Ok(t[1] - t[0]);
    }
    Ok(fs.map(|f| 1.0 / f).unwrap_or(1.0))
}

fn scales_of(scales: &Option<PyReadonlyArray1<f64>>, n: usize, nv: usize, simd: bool) -> Vec<f64> {
    match scales {
        Some(s) => s.as_array().to_vec(),
        None => unsafe {
            // cwt.rs:461-489 (cwt_simd.rs:474-545 when simd)
            let ns = ffi::ssq_cwt_default_scales(n as i64, nv as c_int, simd as c_int, std::ptr::null_mut());
            let mut v = vec![0.0f64; ns.max(0) as usize];
            if ns > 0 {
                ffi::ssq_cwt_default_scales(n as i64, nv as c_int, simd as c_int, v.as_mut_ptr());
            }
            v
        },
    }
}

#[allow(clippy::too_many_arguments)]
fn cwt_impl<'py>(
    py: Python<'py>,
    x: PyReadonlyArray1<f64>,
    wavelet: &str,
    scales: Option<PyReadonlyArray1<f64>>,
    fs: Option<f64>,
    t: Option<PyReadonlyArray1<f64>>,
    nv: usize,
    l1_norm: bool,
    derivative: bool,
    padtype: &str,
    rpadded: bool,
    simd: bool,
) -> PyResult<(PyObject, PyObject, Option<PyObject>)> {
    let x_s = x.as_array().to_owned();
    let n = x_s.len();
    let dt = dt_of(fs, &t)?;
    let sc = scales_of(&scales, n, nv, simd);
    let ns = sc.len();
    let (mut pad_len, mut n1) = (0i64, 0i64);
    let st = unsafe { ffi::ssq_cwt_shape(n as i64, &mut pad_len, &mut n1) }; // cwt.rs:87,98
    ffi::check(st, std::ptr::null())?;
    let cols = if rpadded { pad_len as usize } else { n };
    let mut wx = Array2::<Complex64>::zeros((ns, cols));
    let mut dwx = if derivative { Some(Array2::<Complex64>::zeros((ns, cols))) } else { None };
    let flags = (if l1_norm { 0 } else { ffi::SSQ_FLAG_L2_NORM }) | (if rpadded { ffi::SSQ_FLAG_RPADDED } else { 0 })
        | (if simd { ffi::SSQ_FLAG_SIMD_SCALES } else { 0 });
    let (wav, pad) = (wavelet_code(wavelet), pad_code(padtype));
    if ns > 0 {
        let dptr = dwx.as_mut().map(|d| d.as_mut_ptr() as *mut f64).unwrap_or(std::ptr::null_mut());
        let st = py.allow_threads(|| {
            ffi::with_ctx(|c| unsafe {
                ffi::ssq_cwt_f64(c, x_s.as_ptr(), n as i64, wav, sc.as_ptr(), ns as i64, dt, pad, flags,
                                 wx.as_mut_ptr() as *mut f64, dptr)
            })
        });
        ffi::with_ctx(|c| ffi::check(st, c))?;
    }
    Ok((wx.into_pyarray(py).into_py(py), Array1::from(sc).into_pyarray(py).into_py(py),
        dwx.map(|d| d.into_pyarray(py).into_py(py))))
}

/// cwt.rs:32-144: always a 3-tuple (Wx, scales, dWx | None); `vectorized` / `patience` accepted and unused
#[pyfunction]
#[pyo3(signature = (x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=true, derivative=false, padtype="reflect", rpadded=false, vectorized=true, patience=0))]
#[allow(clippy::too_many_arguments)]
pub fn cwt<'py>(
    py: Python<'py>, x: PyReadonlyArray1<f64>, wavelet: &str, scales: Option<PyReadonlyArray1<f64>>, fs: Option<f64>,
    t: Option<PyReadonlyArray1<f64>>, nv: usize, l1_norm: bool, derivative: bool, padtype: &str, rpadded: bool,
    vectorized: bool, patience: usize,
) -> PyResult<(PyObject, PyObject, Option<PyObject>)> {
    let _ = (vectorized, patience);
    cwt_impl(py, x, wavelet, scales, fs, t, nv, l1_norm, derivative, padtype, rpadded, false)
}

/// cwt_simd.rs:38-66: `cwt` with the exp(p ln 2) default-scale generator
#[pyfunction]
#[pyo3(signature = (x, wavelet="gmw", scales=None, fs=None, t=None, nv=32, l1_norm=true, derivative=false, padtype="reflect", rpadded=false, vectorized=true, patience=0))]
#[allow(clippy::too_many_arguments)]
pub fn cwt_simd<'py>(
    py: Python<'py>, x: PyReadonlyArray1<f64>, wavelet: &str, scales: Option<PyReadonlyArray1<f64>>, fs: Option<f64>,
    t: Option<PyReadonlyArray1<f64>>, nv: usize, l1_norm: bool, derivative: bool, padtype: &str, rpadded: bool,
    vectorized: bool, patience: usize,
) -> PyResult<(PyObject, PyObject, Option<PyObject>)> {
    let _ = (vectorized, patience);
    cwt_impl(py, x, wavelet, scales, fs, t, nv, l1_norm, derivative, padtype, rpadded, true)
}

/// ssq_cwt.rs:245-493; `difftype` / `vectorized` ignored as in the reference (:296-297)
#[pyfunction]
#[pyo3(signature = (x, wavelet="gmw", scales=None, fs=None, t=None, ssq_freqs=None, nv=32, padtype="reflect", squeezing="sum", maprange="peak", difftype="trig", gamma=None, vectorized=true, flipud=true))]
#[allow(clippy::too_many_arguments)]
pub fn ssq_cwt<'py>(
    py: Python<'py>, x: PyReadonlyArray1<f64>, wavelet: &str, scales: Option<PyReadonlyArray1<f64>>, fs: Option<f64>,
    t: Option<PyReadonlyArray1<f64>>, ssq_freqs: Option<&str>, nv: usize, padtype: &str, squeezing: &str, maprange: &str,
    difftype: &str, gamma: Option<f64>, vectorized: bool, flipud: bool,
) -> PyResult<(PyObject, PyObject)> {
    let _ = (difftype, vectorized);
    let x_s = x.as_array().to_owned();
    let n = x_s.len();
    let dt = dt_of(fs, &t)?;
    let sc = scales_of(&scales, n, nv, false);
    let ns = sc.len();
    assert!(ns >= 1, "no scales: index out of bounds (ssq_cwt.rs:459)");
    let mut tx = Array2::<Complex64>::zeros((ns, n));
    let mut sf = Array1::<f64>::zeros(ns);
    let dist = if ssq_freqs == Some("linear") { 1 } else { 0 }; // anything else: log (ssq_cwt.rs:56-112)
    let mr = if maprange == "maximal" { 1 } else { 0 }; // anything else: 1 / scales (ssq_cwt.rs:450-461)
    let (wav, pad, sq) = (wavelet_code(wavelet), pad_code(padtype), squeeze_code(squeezing));
    let flags = if flipud { 0 } else { ffi::SSQ_FLAG_NO_FLIPUD };
    let g = gamma.unwrap_or(f64::NAN);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_ssq_cwt_f64(c, x_s.as_ptr(), n as i64, wav, sc.as_ptr(), ns as i64, dt, dist, pad, sq, mr, g, flags,
                                 tx.as_mut_ptr() as *mut f64, sf.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok((tx.into_pyarray(py).into_py(py), sf.into_pyarray(py).into_py(py)))
}

/// cwt.rs:548-718 (declared in _rs.pyi:62-73, never registered by the reference's lib.rs)
#[pyfunction]
#[pyo3(signature = (wx, wavelet="gmw", scales=None, nv=None, one_int=true, x_len=None, x_mean=0.0, padtype="reflect", rpadded=false, l1_norm=true, exact_adm=false))]
#[allow(clippy::too_many_arguments)]
pub fn icwt<'py>(
    py: Python<'py>, wx: PyReadonlyArray2<Complex64>, wavelet: &str, scales: Option<PyReadonlyArray1<f64>>,
    nv: Option<usize>, one_int: bool, x_len: Option<usize>, x_mean: f64, padtype: &str, rpadded: bool, l1_norm: bool,
    exact_adm: bool,
) -> PyResult<PyObject> {
    let _ = (nv, padtype, rpadded);
    let sc = match scales {
        Some(s) => s.as_array().to_vec(),
        None => return Err(PyValueError::new_err("Scales must be provided")), // cwt.rs:572-575
    };
    let w = wx.as_array().as_standard_layout().to_owned();
    let (ns, ncols) = (w.shape()[0], w.shape()[1]);
    let xl = x_len.unwrap_or(ncols);
    let mut x = Array1::<f64>::zeros(xl);
    let flags = (if l1_norm { 0 } else { ffi::SSQ_FLAG_L2_NORM }) | (if exact_adm { ffi::SSQ_FLAG_ADM_EXACT } else { 0 });
    let wav = wavelet_code(wavelet);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_icwt_f64(c, w.as_ptr() as *const f64, ns as i64, ncols as i64, wav, sc.as_ptr(), one_int as c_int,
                              xl as i64, x_mean, flags, x.as_mut_ptr())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok(x.into_pyarray(py).into_py(py))
}

/// Inversion of `ssq_cwt` (spec old/ssqueezepy/_ssq_cwt.py:313-402): the full inversion, or with `cc`, `cw` the curve
/// bands, [K + 1, n] with the residual last
#[pyfunction]
#[pyo3(signature = (tx, wavelet="gmw", scales=None, cc=None, cw=None))]
pub fn issq_cwt<'py>(
    py: Python<'py>, tx: PyReadonlyArray2<Complex64>, wavelet: &str, scales: Option<PyReadonlyArray1<f64>>,
    cc: Bands<'py>, cw: Bands<'py>,
) -> PyResult<PyObject> {
    let sc = match scales {
        Some(s) => s.as_array().to_vec(),
        None => return Err(PyValueError::new_err("Scales must be provided")),
    };
    let t = tx.as_array().as_standard_layout().to_owned();
    let (ns, n) = (t.shape()[0], t.shape()[1]);
    let wav = wavelet_code(wavelet);
    if let Some((cc, cw, k)) = bands(cc, cw, n)? {
        let mut x = Array2::<f64>::zeros((k + 1, n));
        let st = py.allow_threads(|| {
            ffi::with_ctx(|c| unsafe {
                ffi::ssq_issq_cwt_components_f64(c, t.as_ptr() as *const f64, ns as i64, n as i64, wav, sc.as_ptr(),
                                                 cc.as_ptr(), cw.as_ptr(), k as c_int, x.as_mut_ptr())
            })
        });
        ffi::with_ctx(|c| ffi::check(st, c))?;
        return Ok(x.into_pyarray(py).into_py(py));
    }
    let mut x = Array1::<f64>::zeros(n);
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_issq_cwt_f64(c, t.as_ptr() as *const f64, ns as i64, n as i64, wav, sc.as_ptr(), x.as_mut_ptr())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok(x.into_pyarray(py).into_py(py))
}

/// Css = integral psi-hat(w) / w dw of the wavelet `cwt` / `ssq_cwt` evaluate
#[pyfunction]
#[pyo3(signature = (wavelet="gmw"))]
pub fn adm_ssq(wavelet: &str) -> PyResult<f64> {
    let mut css = 0.0f64;
    let st = unsafe { ffi::ssq_cwt_admissibility(wavelet_code(wavelet), &mut css) };
    ffi::check(st, std::ptr::null())?;
    Ok(css)
}

/// Ridge extraction (rust/src/ridge/{mod,extraction}.rs are empty in the reference; spec
/// old/ssqueezepy/ridge_extraction.py:11-232).  Returns ridge_idxs [n_time, n_ridges].
#[pyfunction]
#[pyo3(signature = (tf, scales, penalty=2.0, n_ridges=1, bw=15, transform="cwt"))]
pub fn extract_ridges<'py>(
    py: Python<'py>, tf: PyReadonlyArray2<Complex64>, scales: PyReadonlyArray1<f64>, penalty: f64, n_ridges: usize,
    bw: usize, transform: &str,
) -> PyResult<PyObject> {
    let t = tf.as_array().as_standard_layout().to_owned();
    let sc = scales.as_array().to_vec();
    let (nf, nt) = (t.shape()[0], t.shape()[1]);
    if sc.len() != nf {
        return Err(PyValueError::new_err("scales must have one entry per row of Tf"));
    }
    let mut idx = Array2::<i32>::zeros((nt, n_ridges));
    let tr = if transform == "cwt" { 0 } else { 1 };
    let st = py.allow_threads(|| {
        ffi::with_ctx(|c| unsafe {
            ffi::ssq_extract_ridges_host(c, t.as_ptr() as *const std::os::raw::c_void, 1, nf as i64, nt as i64, sc.as_ptr(),
                                         penalty, n_ridges as c_int, bw as c_int, tr, idx.as_mut_ptr(),
                                         std::ptr::null_mut(), std::ptr::null_mut(), std::ptr::null_mut())
        })
    });
    ffi::with_ctx(|c| ffi::check(st, c))?;
    Ok(idx.into_pyarray(py).into_py(py))
}

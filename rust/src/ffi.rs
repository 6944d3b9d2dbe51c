// ffi.rs -- the C ABI of libssqcuda (include/ssqcuda.h), one declaration per entry point, plus the per-thread
// context and the status -> Python exception mapping.  Generated from the header (tests/test_rust_crate_sync.py
// checks names and arities against it); the header names the reference interface every entry point replaces.
#![allow(dead_code)]
use std::os::raw::{c_char, c_double, c_float, c_int, c_uint, c_void};

#[repr(C)]
pub struct SsqCtx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct SsqStream {
    _private: [u8; 0],
}
#[repr(C)]
pub struct SsqFeeder {
    _private: [u8; 0],
}
#[repr(C)]
pub struct SsqIstream {
    _private: [u8; 0],
}

pub const SSQ_FLAG_MODULATED: c_uint = 1 << 0;
pub const SSQ_FLAG_NO_FLIPUD: c_uint = 1 << 1;
pub const SSQ_FLAG_L2_NORM: c_uint = 1 << 2;
pub const SSQ_FLAG_RPADDED: c_uint = 1 << 3;
pub const SSQ_FLAG_SIMD_SCALES: c_uint = 1 << 4;
pub const SSQ_FLAG_ADM_EXACT: c_uint = 1 << 5;

extern "C" {
    pub fn ssq_version() -> *const c_char;
    pub fn ssq_hello_from_bin() -> *const c_char;
    pub fn ssq_device_count() -> c_int;
    pub fn ssq_ctx_create(device: c_int, out: *mut *mut SsqCtx) -> c_int;
    pub fn ssq_ctx_destroy(ctx: *mut SsqCtx);
    pub fn ssq_last_error(ctx: *const SsqCtx) -> *const c_char;
    pub fn ssq_ctx_set_stream(ctx: *mut SsqCtx, cuda_stream: *mut c_void) -> c_int;
    pub fn ssq_ctx_synchronize(ctx: *mut SsqCtx) -> c_int;
    pub fn ssq_ctx_set_option(ctx: *mut SsqCtx, name: *const c_char, value: i64) -> c_int;
    pub fn ssq_ctx_launch_count(ctx: *const SsqCtx) -> u64;
    pub fn ssq_ctx_last_kernel_ms(ctx: *mut SsqCtx) -> c_float;
    pub fn ssq_ctx_last_kernel_name(ctx: *const SsqCtx) -> *const c_char;
    pub fn ssq_stft_shape(n: i64, n_fft: c_int, hop: c_int, n_freqs: *mut i64, n_frames: *mut i64) -> c_int;
    pub fn ssq_cwt_shape(n: i64, pad_len: *mut i64, n1: *mut i64) -> c_int;
    pub fn ssq_cwt_default_scales(n: i64, nv: c_int, simd: c_int, scales: *mut c_double) -> i64;
    pub fn ssq_stft_f64(ctx: *mut SsqCtx, x: *const c_double, n: i64, n_fft: c_int, hop: c_int, window: *const c_double, win_n: i64, padtype: c_int, sx: *mut c_double, freqs: *mut c_double) -> c_int;
    pub fn ssq_ssq_stft_f64(ctx: *mut SsqCtx, x: *const c_double, n: i64, window: *const c_double, win_n: i64, n_fft: c_int, win_len: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, flags: c_uint, tx: *mut c_double, ssq_freqs: *mut c_double, sx: *mut c_double, dsx: *mut c_double, w: *mut c_double, kb: *mut i32) -> c_int;
    pub fn ssq_istft_f64(ctx: *mut SsqCtx, sx: *const c_double, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, n: i64, win_exp: c_int, x: *mut c_double) -> c_int;
    pub fn ssq_issq_stft_f64(ctx: *mut SsqCtx, tx: *const c_double, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, y: *mut c_double) -> c_int;
    pub fn ssq_cwt_f64(ctx: *mut SsqCtx, x: *const c_double, n: i64, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, padtype: c_int, flags: c_uint, wx: *mut c_double, dwx: *mut c_double) -> c_int;
    pub fn ssq_ssq_cwt_f64(ctx: *mut SsqCtx, x: *const c_double, n: i64, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, freq_dist: c_int, padtype: c_int, squeezing: c_int, maprange: c_int, gamma: c_double, flags: c_uint, tx: *mut c_double, ssq_freqs: *mut c_double, w: *mut c_double, kb: *mut i32) -> c_int;
    pub fn ssq_icwt_f64(ctx: *mut SsqCtx, wx: *const c_double, ns: i64, n_cols: i64, wavelet: c_int, scales: *const c_double, one_int: c_int, x_len: i64, x_mean: c_double, flags: c_uint, x: *mut c_double) -> c_int;
    pub fn ssq_cwt_admissibility(wavelet: c_int, css: *mut c_double) -> c_int;
    pub fn ssq_issq_cwt_f64(ctx: *mut SsqCtx, tx: *const c_double, ns: i64, n: i64, wavelet: c_int, scales: *const c_double, x: *mut c_double) -> c_int;
    pub fn ssq_issq_cwt_components_f64(ctx: *mut SsqCtx, tx: *const c_double, ns: i64, n: i64, wavelet: c_int, scales: *const c_double, cc: *const c_int, cw: *const c_int, k: c_int, x: *mut c_double) -> c_int;
    pub fn ssq_issq_stft_components_f64(ctx: *mut SsqCtx, tx: *const c_double, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, cc: *const i32, cw: *const i32, k: c_int, y: *mut c_double) -> c_int;
    pub fn ssq_ssq_stft_batch_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, flags: c_uint, d_tx: *mut c_float) -> c_int;
    pub fn ssq_ssq_stft_batch_diag_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, flags: c_uint, d_tx: *mut c_float, d_sx: *mut c_float, d_dsx: *mut c_float, d_w: *mut c_float, d_kb: *mut i32) -> c_int;
    pub fn ssq_stft_batch_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, padtype: c_int, d_sx: *mut c_float) -> c_int;
    pub fn ssq_istft_batch_f32(ctx: *mut SsqCtx, d_sx: *const c_float, channels: i64, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, n_out: i64, win_exp: c_int, d_xout: *mut c_float) -> c_int;
    pub fn ssq_issq_stft_batch_f32(ctx: *mut SsqCtx, d_tx: *const c_float, channels: i64, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, fs: c_double, d_y: *mut c_float) -> c_int;
    pub fn ssq_issq_stft_components_batch_f32(ctx: *mut SsqCtx, d_tx: *const c_float, channels: i64, n_freqs: i64, n_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, fs: c_double, d_cc: *const i32, d_cw: *const i32, k: c_int, d_y: *mut c_float) -> c_int;
    pub fn ssq_cwt_batch_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, padtype: c_int, flags: c_uint, d_wx: *mut c_float, d_dwx: *mut c_float) -> c_int;
    pub fn ssq_ssq_cwt_batch_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, freq_dist: c_int, padtype: c_int, squeezing: c_int, maprange: c_int, gamma: c_double, flags: c_uint, d_tx: *mut c_float, ssq_freqs: *mut c_double) -> c_int;
    pub fn ssq_ssq_cwt_batch_diag_f32(ctx: *mut SsqCtx, d_x: *const c_float, channels: i64, n: i64, x_stride: i64, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, freq_dist: c_int, padtype: c_int, squeezing: c_int, maprange: c_int, gamma: c_double, flags: c_uint, d_tx: *mut c_float, ssq_freqs: *mut c_double, d_w: *mut c_float, d_kb: *mut i32) -> c_int;
    pub fn ssq_icwt_batch_f32(ctx: *mut SsqCtx, d_wx: *const c_float, channels: i64, ns: i64, n_cols: i64, wavelet: c_int, scales: *const c_double, one_int: c_int, x_len: i64, x_mean: c_double, flags: c_uint, d_x: *mut c_float) -> c_int;
    pub fn ssq_issq_cwt_batch_f32(ctx: *mut SsqCtx, d_tx: *const c_float, channels: i64, ns: i64, n: i64, wavelet: c_int, scales: *const c_double, d_x: *mut c_float) -> c_int;
    pub fn ssq_issq_cwt_components_batch_f32(ctx: *mut SsqCtx, d_tx: *const c_float, channels: i64, ns: i64, n: i64, wavelet: c_int, scales: *const c_double, d_cc: *const i32, d_cw: *const i32, k: c_int, d_x: *mut c_float) -> c_int;
    pub fn ssq_wavelet_morlet(kind: c_int, w: *const c_double, n: i64, scale: c_double, mu: c_double, out: *mut c_double) -> c_int;
    pub fn ssq_wavelet_gmw(kind: c_int, w: *const c_double, n: i64, scale: c_double, gamma: c_double, beta: c_double, norm_bandpass: c_int, order: c_int, out: *mut c_double) -> c_int;
    pub fn ssq_wavelet_gmw_center_frequency(gamma: c_double, beta: c_double, kind: c_int, out: *mut c_double) -> c_int;
    pub fn ssq_extract_ridges_batch(ctx: *mut SsqCtx, d_tf: *const c_void, is_f64: c_int, channels: i64, n_freq: i64, n_time: i64, scales: *const c_double, penalty: c_double, n_ridges: c_int, bw: c_int, transform: c_int, d_ridge_idxs: *mut i32, d_ridge_f: *mut c_void, d_ridge_e: *mut c_void, d_e_all: *mut c_void) -> c_int;
    pub fn ssq_extract_ridges_host(ctx: *mut SsqCtx, tf: *const c_void, is_f64: c_int, n_freq: i64, n_time: i64, scales: *const c_double, penalty: c_double, n_ridges: c_int, bw: c_int, transform: c_int, ridge_idxs: *mut i32, ridge_f: *mut c_void, ridge_e: *mut c_void, e_all: *mut c_void) -> c_int;
    pub fn ssq_ssq_stft_host_f32(ctx: *mut SsqCtx, x: *const c_float, channels: i64, n: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, flags: c_uint, tx: *mut c_float) -> c_int;
    pub fn ssq_stft_host_f32(ctx: *mut SsqCtx, x: *const c_float, channels: i64, n: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, padtype: c_int, sx: *mut c_float) -> c_int;
    pub fn ssq_stream_create(ctx: *mut SsqCtx, channels: i64, n_total: i64, max_chunk: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, out: *mut *mut SsqStream) -> c_int;
    pub fn ssq_stream_create_ex(ctx: *mut SsqCtx, channels: i64, n_total: i64, max_chunk: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, fs: c_double, padtype: c_int, squeezing: c_int, gamma: c_double, mode: c_int, flags: c_uint, out: *mut *mut SsqStream) -> c_int;
    pub fn ssq_stream_destroy(s: *mut SsqStream);
    pub fn ssq_stream_total_frames(s: *const SsqStream) -> i64;
    pub fn ssq_stream_frames_after(s: *const SsqStream, n_new: i64) -> i64;
    pub fn ssq_stream_push_i16(s: *mut SsqStream, d_chunk: *const i16, n_new: i64, scale: c_float, d_tx: *mut c_float, frames_written: *mut i64) -> c_int;
    pub fn ssq_stream_push_f32(s: *mut SsqStream, d_chunk: *const c_float, n_new: i64, scale: c_float, d_tx: *mut c_float, frames_written: *mut i64) -> c_int;
    pub fn ssq_stream_create_cwt(ctx: *mut SsqCtx, channels: i64, n_total: i64, max_chunk: i64, block: i64, overlap: i64, mode: c_int, wavelet: c_int, scales: *const c_double, ns: i64, dt: c_double, freq_dist: c_int, padtype: c_int, squeezing: c_int, maprange: c_int, gamma: c_double, flags: c_uint, out: *mut *mut SsqStream) -> c_int;
    pub fn ssq_stream_ssq_freqs(s: *const SsqStream, last_block: c_int, out: *mut c_double) -> c_int;
    pub fn ssq_feeder_create(s: *mut SsqStream, dtype: c_int, depth: c_int, out: *mut *mut SsqFeeder) -> c_int;
    pub fn ssq_feeder_destroy(f: *mut SsqFeeder);
    pub fn ssq_feeder_push(f: *mut SsqFeeder, h_chunk: *const c_void, n_new: i64, scale: c_float, d_tx: *mut c_float, frames_written: *mut i64) -> c_int;
    pub fn ssq_istream_create(ctx: *mut SsqCtx, channels: i64, n_frames_total: i64, n_out: i64, max_frames: i64, window: *const c_double, win_n: i64, n_fft: c_int, hop: c_int, win_exp: c_int, mode: c_int, fs: c_double, out_format: c_int, out: *mut *mut SsqIstream) -> c_int;
    pub fn ssq_istream_destroy(s: *mut SsqIstream);
    pub fn ssq_istream_total_samples(s: *const SsqIstream) -> i64;
    pub fn ssq_istream_samples_after(s: *const SsqIstream, n_new: i64) -> i64;
    pub fn ssq_istream_push(s: *mut SsqIstream, d_sx: *const c_float, n_new: i64, scale: c_float, d_out: *mut c_void, samples_written: *mut i64) -> c_int;
    pub fn ssq_host_alloc(p: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn ssq_host_free(p: *mut c_void);
    pub fn ssq_memcpy_async(dst: *mut c_void, src: *const c_void, bytes: usize, kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn ssq_device_numa_node(device: c_int, node: *mut c_int) -> c_int;
    pub fn ssq_host_alloc_near(p: *mut *mut c_void, bytes: usize, device: c_int) -> c_int;
}

thread_local! {
    // One context per host thread: contexts are not thread-safe, the reference's functions are re-entrant and release
    // the GIL (stft.rs:37, ssq_stft.rs:122, cwt.rs:85, ssq_cwt.rs:329).
    pub static CTX: *mut SsqCtx = unsafe {
        let mut c = std::ptr::null_mut();
        let dev = std::env::var("SSQ_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        if ssq_ctx_create(dev, &mut c) != 0 { std::ptr::null_mut() } else { c }
    };
}

/// Status -> PyErr.  SSQ_EINVAL is the reference's PyValueError (ssq_stft.rs:96-101, cwt.rs:68-70); SSQ_EPANIC marks an
/// input on which the reference panics (PanicException): panic here too.  There is no CPU fallback: without a device
/// every call fails with SSQ_ECUDA -> RuntimeError.
pub fn check(status: c_int, ctx: *const SsqCtx) -> pyo3::PyResult<()> {
    use pyo3::exceptions::{PyMemoryError, PyRuntimeError, PyValueError};
    if status == 0 {
        return Ok(());
    }
    let msg = unsafe { std::ffi::CStr::from_ptr(ssq_last_error(ctx)) }.to_string_lossy().into_owned();
    Err(match status {
        1 => PyValueError::new_err(msg),
        3 => PyMemoryError::new_err(msg),
        5 => panic!("{msg}"),
        _ => PyRuntimeError::new_err(msg),
    })
}

pub fn with_ctx<R>(f: impl FnOnce(*mut SsqCtx) -> R) -> R {
    CTX.with(|c| f(*c))
}

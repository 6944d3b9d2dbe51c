/* ssqcuda.h -- C ABI of libssqcuda: the B200 (sm_100a) replacement for the
 * compute path behind the reference's `ssqueeze._rs` pyo3 module.
 *
 * Drop-in boundary.  The reference's FFI for this path is the set of
 * #[pyfunction]s registered in rust/src/lib.rs:23-35.  A maintainer keeps the
 * pyo3 host crate and replaces each function body (everything inside
 * `Python::allow_threads`) by one call into this library; INTEGRATION.md shows
 * the `extern "C"` block and the rewritten bodies.  Each entry point below
 * names the reference interface it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; complex arrays are interleaved (re, im);
 *  - every function returns an ssq_status; nothing throws or aborts across
 *    the ABI; `ssq_last_error(ctx)` gives the message of the last failure on
 *    that context (`ssq_last_error(NULL)`: last failure of a call that had no
 *    context, thread-local);
 *  - the caller allocates all outputs; sizes come from the *_shape queries;
 *  - a context is bound to one CUDA device and is NOT thread-safe; use one
 *    context per thread/device (the reference's functions are re-entrant and
 *    release the GIL: stft.rs:37, ssq_stft.rs:122, cwt.rs:85, ssq_cwt.rs:329);
 *  - `*_f64` entry points take/return HOST buffers with the reference's dtypes
 *    (float64 / complex128); arithmetic on the device is fp32;
 *  - `*_batch_f32` entry points take/return DEVICE (or pinned-host mapped)
 *    buffers: x[channels, n] fp32 C-contiguous in, complex64 out
 *    [channels, rows, cols]; they are asynchronous on the context's stream;
 *  - `*_host_f32` entry points take HOST buffers (pinned preferred) and do the
 *    host<->device copies themselves (synchronous at return);
 *  - streams (`ssq_stream_*` forward, `ssq_istream_*` inverse) take a long
 *    recording chunk by chunk and are exact at chunk seams; they own their
 *    buffers, so calls on the same context between two pushes are allowed;
 *    the CWT streams (`ssq_stream_create_cwt`) are blockwise with an overlap,
 *    as the reference's dask caller is, and independent of how the recording
 *    is cut into pushes;
 *  - there is no CPU fallback: without a usable CUDA device every compute
 *    call fails with SSQ_ECUDA.
 */
#ifndef SSQCUDA_H
#define SSQCUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ssq_ctx ssq_ctx;

typedef enum ssq_status {
  SSQ_OK = 0,
  SSQ_EINVAL = 1,        /* maps to PyValueError (ssq_stft.rs:96-101, cwt.rs:68-70) */
  SSQ_ECUDA = 2,         /* CUDA runtime / launch failure, or no device */
  SSQ_ENOMEM = 3,        /* device or host allocation failed */
  SSQ_EUNSUPPORTED = 4,  /* valid in the reference, not built here (yet) */
  SSQ_EPANIC = 5         /* input on which the reference panics (PanicException) */
} ssq_status;

/* padtype: the reference matches "reflect" | "zero" and silently falls back to
 * reflect for anything else (stft.rs:25-29, ssq_stft.rs:124-128, cwt.rs:88-92) */
enum { SSQ_PAD_REFLECT = 0, SSQ_PAD_ZERO = 1 };
/* squeezing: "sum" | "lebesgue", fallback sum (ssq_stft.rs:292-296, ssq_cwt.rs:199-206) */
enum { SSQ_SQUEEZE_SUM = 0, SSQ_SQUEEZE_LEBESGUE = 1 };
/* wavelet: "morlet", anything else is GMW(gamma=3, beta=60) (cwt.rs:496-541) */
enum { SSQ_WAVELET_GMW = 0, SSQ_WAVELET_MORLET = 1 };
/* maprange: "maximal", anything else uses 1/scales (ssq_cwt.rs:450-461) */
enum { SSQ_MAPRANGE_PEAK = 0, SSQ_MAPRANGE_MAXIMAL = 1 };
/* ssq_freqs distribution: "linear", anything else log (ssq_cwt.rs:56-112) */
enum { SSQ_FREQS_LOG = 0, SSQ_FREQS_LINEAR = 1 };

/* flags (bit set) */
enum {
  SSQ_FLAG_MODULATED = 1u << 0,  /* ssq_stft: multiply Sx by exp(+2 pi i k (n_fft/2)/n_fft) before squeezing
                                    (build-side extension needed by issq_stft; SURVEY 8a row 10) */
  SSQ_FLAG_NO_FLIPUD = 1u << 1,  /* ssq_cwt: flipud=false (ssq_cwt.rs:180-184) */
  SSQ_FLAG_L2_NORM = 1u << 2,    /* cwt: l1_norm=false -> multiply rows by sqrt(scale) (cwt.rs:253) */
  SSQ_FLAG_RPADDED = 1u << 3,    /* cwt: return the padded [ns, pad_len] rows (cwt.rs:108-110) */
  SSQ_FLAG_SIMD_SCALES = 1u << 4, /* cwt_simd default-scale generator (cwt_simd.rs:489-527) */
  SSQ_FLAG_ADM_EXACT = 1u << 5    /* icwt: divide by the wavelet's true admissibility integral
                                     (ssq_cwt_admissibility) instead of the reference's placeholders
                                     0.776 / 1.0 (cwt.rs:579-583), so that cwt -> icwt reconstructs x */
};

/* ---- library / context ------------------------------------------------- */
/* library identification string */
const char* ssq_version(void);
/* replaces hello_from_bin (lib.rs:16-19): the reference's greeting, verbatim */
const char* ssq_hello_from_bin(void);
int ssq_device_count(void);
ssq_status ssq_ctx_create(int device, ssq_ctx** out);
void ssq_ctx_destroy(ssq_ctx* ctx);
const char* ssq_last_error(const ssq_ctx* ctx);
/* borrow a caller-owned cudaStream_t (NULL restores the context's own stream) */
ssq_status ssq_ctx_set_stream(ssq_ctx* ctx, void* cuda_stream);
ssq_status ssq_ctx_synchronize(ssq_ctx* ctx);
/* context options (DESIGN.md 6c); an unknown name returns SSQ_EINVAL.  Nothing reads them from the environment.
 * Reference paths for cross-checks, none changes results beyond fp32 rounding: no_h32r, no_r1024, no_r256 (n_fft
 * 512 / 1024 / 256 through the generic shared-memory kernels), no_cwt_fused (ssq_cwt through the ordered,
 * bit-deterministic stand-alone reassignment).
 * One option does change results: upstream_framing = 1 frames the STFT family as upstream ssqueezepy does (left pad
 * n_fft / 2 instead of the crate's (n_fft - 1) / 2, stft_utils.rs:22) -- the upstream-compatible mode, SURVEY 8f rank 3. */
ssq_status ssq_ctx_set_option(ssq_ctx* ctx, const char* name, int64_t value);
/* number of kernels this context has launched since creation (bench "gpu_launches") */
uint64_t ssq_ctx_launch_count(const ssq_ctx* ctx);
/* device-time of the most recent batch call's dominant kernel, measured with
 * CUDA events on the context's stream (ms); < 0 when not available */
float ssq_ctx_last_kernel_ms(ssq_ctx* ctx);
/* name of that kernel (static string; "" before the first call) */
const char* ssq_ctx_last_kernel_name(const ssq_ctx* ctx);

/* ---- shape queries ------------------------------------------------------ */
/* stft.rs:32-34 / ssq_stft.rs:182-184: n_freqs = n_fft/2+1,
 * n_frames = (n + n_fft-1 - n_fft)/hop + 1 = (n-1)/hop + 1 */
ssq_status ssq_stft_shape(int64_t n, int n_fft, int hop, int64_t* n_freqs, int64_t* n_frames);
/* cwt.rs:87,98 / ssq_cwt.rs:331,353: pad_len = next_pow2(n + n/2), n1 = (pad_len-n)/2 */
ssq_status ssq_cwt_shape(int64_t n, int64_t* pad_len, int64_t* n1);
/* cwt.rs:461-489 (and cwt_simd.rs:474-545 when simd != 0): returns the number
 * of default scales; fills `scales` when non-NULL */
int64_t ssq_cwt_default_scales(int64_t n, int nv, int simd, double* scales);

/* ---- reference-typed entry points (host float64 / complex128) ----------- */
/* replaces the body of `stft` (stft.rs:12-95).
 * Sx: complex128 [n_freqs, n_frames] C-order; freqs: float64 [n_freqs]. */
ssq_status ssq_stft_f64(ssq_ctx* ctx, const double* x, int64_t n, int n_fft, int hop,
                        const double* window, int64_t win_n, int padtype,
                        double* Sx, double* freqs);

/* replaces the body of `ssq_stft` (ssq_stft.rs:74-313).  n_fft<=0: min(n,512)
 * (:92); win_len<=0: win_n (:93); gamma NaN ("not given"): 10*EPS64 (:258-261), gamma < 0: nothing is gated (:23).
 * Tx: complex128 [n_freqs, n_frames]; ssq_freqs: float64 [n_freqs].
 * Optional diagnostics (may be NULL), written by the SAME kernel that produces Tx (a compile-time variant
 * with the extra stores): Sx, dSx complex128 same shape; w float64 same shape (+inf where gated);
 * kb int32 same shape: the destination bin of every (source bin, frame), -1 where gated -- what the
 * parity tests compare with the reference's arg-min (ssq_stft.rs:276-301). */
ssq_status ssq_ssq_stft_f64(ssq_ctx* ctx, const double* x, int64_t n,
                            const double* window, int64_t win_n, int n_fft, int win_len,
                            int hop, double fs, int padtype, int squeezing, double gamma,
                            unsigned flags, double* Tx, double* ssq_freqs,
                            double* Sx, double* dSx, double* w, int32_t* kb);

/* `istft`: absent from the Rust crate (lib.rs:25-32) but named by the north
 * star; specified from old/ssqueezepy/_stft.py:184-256 in the Rust framing
 * (unmodulated, pad offset (n_fft-1)/2).  Sx complex128 [n_freqs, n_frames]
 * -> x float64 [n_out], n_out = N if N>0 else hop*n_frames. */
ssq_status ssq_istft_f64(ssq_ctx* ctx, const double* Sx, int64_t n_freqs, int64_t n_frames,
                         const double* window, int64_t win_n, int n_fft, int hop,
                         int64_t N, int win_exp, double* x);

/* `issq_stft` (old/ssqueezepy/_ssq_stft.py:139-198, full inverse; hop must be 1):
 * y[j] = sum_k Re Tx[k,j] * 2 / (window_fit[n_fft/2] * fs). */
ssq_status ssq_issq_stft_f64(ssq_ctx* ctx, const double* Tx, int64_t n_freqs, int64_t n_frames,
                             const double* window, int64_t win_n, int n_fft, int hop,
                             double fs, double* y);

/* replaces the bodies of `cwt` / `cwt_simd` (cwt.rs:46-144, cwt_simd.rs:52-...).
 * scales: float64 [ns] (caller passes the defaults from ssq_cwt_default_scales
 * when the Python argument is None); dt from t[1]-t[0] | 1/fs | 1 (cwt.rs:66-76).
 * Wx / dWx: complex128 [ns, n] (or [ns, pad_len] with SSQ_FLAG_RPADDED);
 * dWx may be NULL (derivative=false). */
ssq_status ssq_cwt_f64(ssq_ctx* ctx, const double* x, int64_t n, int wavelet,
                       const double* scales, int64_t ns, double dt, int padtype,
                       unsigned flags, double* Wx, double* dWx);

/* replaces the body of `ssq_cwt` (ssq_cwt.rs:261-493).
 * Tx complex128 [ns, n]; ssq_freqs float64 [ns] (not flipped, :482).  gamma: NaN = not given (10*EPS64).
 * Optional diagnostics (may be NULL), written by the reassignment itself: w float64 [ns, n] (the phase transform,
 * +inf where gated), kb int32 [ns, n]: the Tx row every (scale, column) was added to, -1 where nothing was added
 * (gated, w not finite, bin outside the grid: ssq_cwt.rs:165-190). */
ssq_status ssq_ssq_cwt_f64(ssq_ctx* ctx, const double* x, int64_t n, int wavelet,
                           const double* scales, int64_t ns, double dt, int freq_dist,
                           int padtype, int squeezing, int maprange, double gamma,
                           unsigned flags, double* Tx, double* ssq_freqs, double* w, int32_t* kb);

/* `icwt` (SURVEY 8f rank 2): cwt.rs:548-718, a #[pyfunction] the reference module never registers.
 * One-integral branch (:590-627, the default): x[j] = (2/adm) dj sum_i Re Wx[i,j] norm_i + x_mean.
 * one_int == 0 (two-integral branch, :629-712: per scale FFT(Wx[i, :x_len]) conj(psi-hat_i) -> IFFT / x_len / scale,
 * summed in the frequency domain here, one inverse transform): any x_len <= n_cols (Bluestein for lengths that are
 * not powers of two).
 * Wx complex128 [ns, n_cols] -> x float64 [x_len] (x_len <= 0: n_cols).
 * flags: SSQ_FLAG_L2_NORM, SSQ_FLAG_ADM_EXACT. */
ssq_status ssq_icwt_f64(ssq_ctx* ctx, const double* Wx, int64_t ns, int64_t n_cols, int wavelet,
                        const double* scales, int one_int, int64_t x_len, double x_mean, unsigned flags,
                        double* x);

/* Css = integral psi-hat(w)/w dw of the wavelet ssq_cwt/cwt evaluate (cwt.rs:492-547; definition
 * old/ssqueezepy/utils/cwt_utils.py:28-47).  Host-side, double. */
ssq_status ssq_cwt_admissibility(int wavelet, double* css);

/* `issq_cwt` (SURVEY 8f rank 2; spec old/ssqueezepy/_ssq_cwt.py:313-378, full inversion):
 * x[j] = (2/Css) dj sum_k Re Tx[k,j], dj = ln(scales[1]/scales[0]) (0.1 if not ascending, as icwt).
 * The dj factor is upstream's `const` (ln 2 / nv), which the reference's ssqueeze leaves out of Tx
 * (ssq_cwt.rs:116-222).  Tx complex128 [ns, n] -> x float64 [n]. */
ssq_status ssq_issq_cwt_f64(ssq_ctx* ctx, const double* Tx, int64_t ns, int64_t n, int wavelet,
                            const double* scales, double* x);

/* `issq_cwt` with curve bands (old/ssqueezepy/_ssq_cwt.py:313-402): component c of column j sums Re Tx over the rows
 * lower .. upper (inclusive), upper = clip(cc[j][c] + cw[j][c], 0, ns), lower = clip(cc[j][c] - cw[j][c], 0, ns)
 * (in 64 bits; cc == -1: no curve at that column); each component is summed from the original Tx, so bands may
 * overlap; the last output row is the residual (rows no band covers).  cc, cw: int32 [n][K], 1 <= K <= 16
 * (SSQ_EUNSUPPORTED otherwise).  x: float64 [K + 1][n]. */
ssq_status ssq_issq_cwt_components_f64(ssq_ctx* ctx, const double* Tx, int64_t ns, int64_t n, int wavelet,
                                       const double* scales, const int* cc, const int* cw, int K, double* x);
/* `issq_stft` with curve bands (upstream's issq_stft(Tx, ..., cc, cw), old/ssqueezepy/_ssq_stft.py:139-198): the
 * bands of ssq_issq_cwt_components_f64 over the n_freqs rows, times 2 / (window_fit[n_fft/2] * fs); hop must be 1.
 * Tx complex128 [n_freqs, n_frames]; cc, cw int32 [n_frames][K]; y float64 [K + 1][n_frames], row K the residual. */
ssq_status ssq_issq_stft_components_f64(ssq_ctx* ctx, const double* Tx, int64_t n_freqs, int64_t n_frames,
                                        const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                        const int32_t* cc, const int32_t* cw, int K, double* y);

/* ---- batched throughput path (device buffers, fp32 / complex64) ---------- */
/* replaces the per-channel Python loop around `_rs.ssq_stft`
 * (tests/stft_ssq_test.py:230-251).  d_x: [channels, n] fp32 with row stride
 * x_stride (elements).  d_Tx: complex64 [channels, n_freqs, n_frames].
 * window is a HOST float64 array (fit to n_fft as ssq_stft.rs:104-119).
 * Asynchronous on the context's stream. */
ssq_status ssq_ssq_stft_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                  int64_t x_stride, const double* window, int64_t win_n,
                                  int n_fft, int hop, double fs, int padtype, int squeezing,
                                  double gamma, unsigned flags, float* d_Tx);
/* diagnostic twin (parity tests, bench.py's parity leg): the same kernel selection; any non-NULL d_Sx / d_dSx
 * (complex64), d_w (fp32, Hz, +inf where gated), d_kb (int32 destination bin per (source bin, frame), -1 gated),
 * each [channels, n_freqs, n_frames], is written by the kernel that produces d_Tx (compile-time variant). */
ssq_status ssq_ssq_stft_batch_diag_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                       int64_t x_stride, const double* window, int64_t win_n,
                                       int n_fft, int hop, double fs, int padtype, int squeezing,
                                       double gamma, unsigned flags, float* d_Tx, float* d_Sx, float* d_dSx,
                                       float* d_w, int32_t* d_kb);
/* same framing, output Sx (complex64 [channels, n_freqs, n_frames]); the
 * window is used as given when win_n >= n_fft (first n_fft taps, stft_utils.rs:8) */
ssq_status ssq_stft_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                              int64_t x_stride, const double* window, int64_t win_n,
                              int n_fft, int hop, int padtype, float* d_Sx);
/* d_Sx complex64 [channels, n_freqs, n_frames] -> d_xout fp32 [channels, n_out] */
ssq_status ssq_istft_batch_f32(ssq_ctx* ctx, const float* d_Sx, int64_t channels,
                               int64_t n_freqs, int64_t n_frames, const double* window,
                               int64_t win_n, int n_fft, int hop, int64_t n_out, int win_exp,
                               float* d_xout);
ssq_status ssq_issq_stft_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels,
                                   int64_t n_freqs, int64_t n_frames, const double* window,
                                   int64_t win_n, int n_fft, double fs, float* d_y);
/* same bands as ssq_issq_cwt_components_batch_f32 on an issq_stft map (hop 1, modulated Tx), times the factor of
 * ssq_issq_stft_batch_f32: d_Tx complex64 [channels, n_freqs, n_frames]; d_cc, d_cw DEVICE int32
 * [channels, n_frames, K]; d_y fp32 [channels, K + 1, n_frames], row K the residual */
ssq_status ssq_issq_stft_components_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels,
                                              int64_t n_freqs, int64_t n_frames, const double* window,
                                              int64_t win_n, int n_fft, double fs, const int32_t* d_cc,
                                              const int32_t* d_cw, int K, float* d_y);
/* d_Wx / d_dWx complex64 [channels, ns, n] (d_dWx may be NULL) */
ssq_status ssq_cwt_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                             int64_t x_stride, int wavelet, const double* scales, int64_t ns,
                             double dt, int padtype, unsigned flags, float* d_Wx, float* d_dWx);
/* d_Tx complex64 [channels, ns, n]; ssq_freqs (host, float64 [ns]) may be NULL */
ssq_status ssq_ssq_cwt_batch_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                 int64_t x_stride, int wavelet, const double* scales,
                                 int64_t ns, double dt, int freq_dist, int padtype,
                                 int squeezing, int maprange, double gamma, unsigned flags,
                                 float* d_Tx, double* ssq_freqs);

/* diagnostic twin: d_w fp32, d_kb int32, each [channels, ns, n] (may be NULL) */
ssq_status ssq_ssq_cwt_batch_diag_f32(ssq_ctx* ctx, const float* d_x, int64_t channels, int64_t n,
                                      int64_t x_stride, int wavelet, const double* scales,
                                      int64_t ns, double dt, int freq_dist, int padtype,
                                      int squeezing, int maprange, double gamma, unsigned flags,
                                      float* d_Tx, double* ssq_freqs, float* d_w, int32_t* d_kb);

/* d_Wx complex64 [channels, ns, n_cols] -> d_x fp32 [channels, x_len] */
ssq_status ssq_icwt_batch_f32(ssq_ctx* ctx, const float* d_Wx, int64_t channels, int64_t ns, int64_t n_cols,
                              int wavelet, const double* scales, int one_int, int64_t x_len, double x_mean,
                              unsigned flags, float* d_x);

/* d_Tx complex64 [channels, ns, n] -> d_x fp32 [channels, n] */
ssq_status ssq_issq_cwt_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels, int64_t ns, int64_t n,
                                  int wavelet, const double* scales, float* d_x);
/* curve bands on the device (the rule of ssq_issq_cwt_components_f64, clipped by the kernel): d_Tx complex64
 * [channels, ns, n]; d_cc, d_cw DEVICE int32 [channels, n, K] (the layout of ssq_extract_ridges_batch's
 * d_ridge_idxs), 1 <= K <= 16; d_x fp32 [channels, K + 1, n], row K the residual.  Channel c equals the one-channel
 * call bit for bit, and one band covering every row equals ssq_issq_cwt_batch_f32 bit for bit. */
ssq_status ssq_issq_cwt_components_batch_f32(ssq_ctx* ctx, const float* d_Tx, int64_t channels, int64_t ns,
                                             int64_t n, int wavelet, const double* scales, const int32_t* d_cc,
                                             const int32_t* d_cw, int K, float* d_x);

/* ---- wavelet generators (SURVEY 8f rank 2) --------------------------------------------------------------
 * The functions src/ssqueeze/_rs.pyi:91-132 declares: `morlet`, `morlet_freq`, `morlet_time` (rust/src/wavelets/
 * morlet.rs:59-146), `gmw`, `gmw_freq`, `gmw_time`, `gmw_center_frequency` (gmw.rs:226-358).  Host arithmetic in
 * double (they are O(n)); no device is needed.  kind: 0 = psi-hat at the given w[n]; 1 = psi-hat on xifn(scale, n)
 * (base.rs:18-33; `w` unused); 2 = the time-domain wavelet (psi-hat (-1)^i, Nyquist bin halved for even n, inverse
 * DFT / n).  out: complex128 [n]. */
ssq_status ssq_wavelet_morlet(int kind, const double* w, int64_t n, double scale, double mu, double* out);
/* norm_bandpass: norm.to_lowercase() == "bandpass" (anything else is the L2 / "energy" normalisation, gmw.rs:44-52);
 * with kind 0 the argument checks of `gmw` apply (SSQ_EINVAL: gamma <= 0, beta < 0, order < 0; gmw.rs:238-246) */
ssq_status ssq_wavelet_gmw(int kind, const double* w, int64_t n, double scale, double gamma, double beta,
                           int norm_bandpass, int order, double* out);
/* kind: 0 "peak" = (beta/gamma)^(1/gamma), 1 "energy" (gmw.rs:331-357) */
ssq_status ssq_wavelet_gmw_center_frequency(double gamma, double beta, int kind, double* out);

/* ---- ridge extraction on a time-frequency map (SURVEY 8f rank 4) --------------------------------------------
 * The reference crate declares rust/src/ridge/{mod,extraction}.rs and leaves them empty; the specification is
 * upstream's forward/backward penalised ridge tracking, old/ssqueezepy/ridge_extraction.py:11-232 (sequential
 * semantics).  Consumes Tx / Wx / Sx where it lies in HBM: only [n_time, n_ridges] indices have to leave the device.
 * d_Tf: complex64 (is_f64 = 0: float arithmetic, eps = EPS32, as upstream does for complex64) or complex128
 * [channels, n_freq, n_time]; scales: host float64 [n_freq] (the second argument of upstream's extract_ridges);
 * transform: 0 'cwt' (penalty on log(scales)), 1 'stft' (on scales); d_ridge_idxs int32 [channels, n_time, n_ridges];
 * d_ridge_f / d_ridge_e (optional, real type of Tf, same shape): scales / energies along the ridges;
 * d_E_all (optional diagnostic, [channels, n_ridges, n_freq, n_time]): -log(energy / max + eps) of every ridge. */
ssq_status ssq_extract_ridges_batch(ssq_ctx* ctx, const void* d_Tf, int is_f64, int64_t channels, int64_t n_freq,
                                    int64_t n_time, const double* scales, double penalty, int n_ridges, int bw,
                                    int transform, int32_t* d_ridge_idxs, void* d_ridge_f, void* d_ridge_e,
                                    void* d_E_all);
/* one map in HOST memory (complex64 or complex128 [n_freq, n_time]); outputs in host memory */
ssq_status ssq_extract_ridges_host(ssq_ctx* ctx, const void* Tf, int is_f64, int64_t n_freq, int64_t n_time,
                                   const double* scales, double penalty, int n_ridges, int bw, int transform,
                                   int32_t* ridge_idxs, void* ridge_f, void* ridge_e, void* E_all);

/* ---- batched path with HOST buffers (copies inside; synchronous) --------- */
/* x: host fp32 [channels, n]; Tx: host complex64 [channels, n_freqs, n_frames] */
ssq_status ssq_ssq_stft_host_f32(ssq_ctx* ctx, const float* x, int64_t channels, int64_t n,
                                 const double* window, int64_t win_n, int n_fft, int hop,
                                 double fs, int padtype, int squeezing, double gamma,
                                 unsigned flags, float* Tx);

/* the same pipeline for `stft` (stft.rs:12-95): Sx host complex64 [channels, n_fft/2+1, n_frames] */
ssq_status ssq_stft_host_f32(ssq_ctx* ctx, const float* x, int64_t channels, int64_t n, const double* window,
                             int64_t win_n, int n_fft, int hop, int padtype, float* Sx);

/* ---- streaming ssq_stft over chunks of an interleaved recording ------------ */
/* replaces the dask map_overlap caller of the reference (tests/stft_ssq_test.py:218-283:
 * (samples, channels) chunks with depth n_fft, a per-channel Python loop inside each chunk).
 * A stream is created for a recording of n_total samples x channels; every push hands over
 * the next chunk as a DEVICE array [n_new, channels] (channels fastest) of int16 or float32,
 * multiplied by `scale` on conversion, and writes the frames that became complete:
 * d_Tx complex64 [channels, n_freqs, frames], frames = ssq_stream_frames_after(s, n_new)
 * queried BEFORE the push.  Exact at chunk seams (padding only at the two ends of the
 * recording): the concatenation over pushes equals ssq_ssq_stft_batch_f32 on the whole signal. */
typedef struct ssq_stream ssq_stream;
ssq_status ssq_stream_create(ssq_ctx* ctx, int64_t channels, int64_t n_total, int64_t max_chunk,
                             const double* window, int64_t win_n, int n_fft, int hop, double fs,
                             int padtype, int squeezing, double gamma, ssq_stream** out);
/* the same with the transform chosen: mode 0 = ssq_stft (flags: SSQ_FLAG_MODULATED), mode 1 = stft (the dask caller of
 * tests/stft_test.py:215-271; the window's first n_fft taps as stft.rs:47-78 takes them; fs, squeezing, gamma unused) */
ssq_status ssq_stream_create_ex(ssq_ctx* ctx, int64_t channels, int64_t n_total, int64_t max_chunk,
                                const double* window, int64_t win_n, int n_fft, int hop, double fs,
                                int padtype, int squeezing, double gamma, int mode, unsigned flags,
                                ssq_stream** out);
void ssq_stream_destroy(ssq_stream* s);
int64_t ssq_stream_total_frames(const ssq_stream* s);
int64_t ssq_stream_frames_after(const ssq_stream* s, int64_t n_new);
ssq_status ssq_stream_push_i16(ssq_stream* s, const int16_t* d_chunk, int64_t n_new, float scale,
                               float* d_Tx, int64_t* frames_written);
ssq_status ssq_stream_push_f32(ssq_stream* s, const float* d_chunk, int64_t n_new, float scale,
                               float* d_Tx, int64_t* frames_written);

/* CWT streams (DESIGN §3.6b): the dask map_overlap(depth=overlap, boundary="reflect") caller of the reference's CWT
 * scripts (tests/cwt_test.py:117-119,187-193), computed on the device from the carry-over buffer.  Block b covers
 * output columns [b block, min((b + 1) block, n_total)); it is the reference's call (mode 2: cwt -> Wx with
 * SSQ_FLAG_L2_NORM as in ssq_cwt_batch_f32; mode 3: ssq_cwt -> Tx with SSQ_FLAG_NO_FLIPUD as in
 * ssq_ssq_cwt_batch_f32) on e_b[j] = x~[b block - overlap + j], j < len_b + 2 overlap, trimmed to columns
 * [overlap, overlap + len_b); x~ mirrors the recording with the edge sample repeated (np.pad mode "symmetric").  The
 * scales are the same for every block; maprange maximal uses each block's own length (ssq_stream_ssq_freqs).  A block
 * is ready once min(n_total, (b + 1) block + overlap) samples have arrived; a push writes every block that became
 * ready: d_Tx complex64 [channels, ns, cols], cols = ssq_stream_frames_after(s, n_new) queried before the push;
 * ssq_stream_total_frames is n_total.  The output does not depend on how the recording is cut into pushes.
 * 1 <= block, 0 <= overlap <= min(block, n_total); the arguments are checked before ctx.  Pushes and the feeder are
 * those of the STFT streams. */
ssq_status ssq_stream_create_cwt(ssq_ctx* ctx, int64_t channels, int64_t n_total, int64_t max_chunk, int64_t block,
                                 int64_t overlap, int mode, int wavelet, const double* scales, int64_t ns, double dt,
                                 int freq_dist, int padtype, int squeezing, int maprange, double gamma,
                                 unsigned flags, ssq_stream** out);
/* the ssq grid of an ssq_cwt stream (float64 [ns]): of the full blocks (last_block = 0) or of the last block, whose
 * grid differs under maprange maximal when it is shorter */
ssq_status ssq_stream_ssq_freqs(const ssq_stream* s, int last_block, double* out);

/* Host feeder of a stream: the chunk pointer is HOST memory (pageable is fine: a memory-mapped (samples, channels)
 * .dat / .bin as the reference's scripts read them, tests/stft_ssq_test.py:218-283, tests/stft_test.py:374-377).
 * dtype 0 = int16, 1 = float32; `depth` (2..8) pinned + device staging slots of max_chunk x channels elements: the
 * host copy of chunk i+1 overlaps the H2D copy of chunk i and the transform of chunk i-1.  ssq_feeder_push queues the
 * work and returns; d_Tx (device, as in ssq_stream_push_*) is written in the order of the context's stream.  The
 * feeder must be destroyed before its stream. */
typedef struct ssq_feeder ssq_feeder;
ssq_status ssq_feeder_create(ssq_stream* s, int dtype, int depth, ssq_feeder** out);
void ssq_feeder_destroy(ssq_feeder* f);
ssq_status ssq_feeder_push(ssq_feeder* f, const void* h_chunk, int64_t n_new, float scale, float* d_Tx,
                           int64_t* frames_written);

/* ---- streaming inverse over chunks of frames (DESIGN §3.4c) ------------------ */
/* The inverse of ssq_stream_*: a stream is created for n_frames_total frames of channels channels; every push hands
 * over the next n_new (<= max_frames) frames as DEVICE complex64 d_Sx [channels, n_freqs, n_new] -- the layout a
 * forward push writes, masked or not -- and writes the output samples that became final to d_out,
 * samples = ssq_istream_samples_after(s, n_new) queried BEFORE the push.  Over all pushes exactly
 * ssq_istream_total_samples(s) samples are written, equal to the batch call on the whole Sx.
 * mode 0 = istft (old/ssqueezepy/_stft.py:184-256, ssq_istft_batch_f32's framing and win_exp; n_out <= 0 means
 * hop * n_frames_total; frames past the batch call's max_hops are accepted and dropped), mode 1 = issq_stft (hop must
 * be 1; Tx computed with SSQ_FLAG_MODULATED; fs as ssq_issq_stft_batch_f32; one sample per frame).
 * out_format 0 = fp32 [channels, samples], 1 = fp32 [samples, channels], 2 = int16 [samples, channels] (round to
 * nearest even, saturated).  Samples are multiplied by (float)(1.0 / scale): scale = 0.195 returns the int16 counts
 * that a forward stream pushed with scale = 0.195 turned into uV.  The stream owns its buffers: a batch call on the
 * same context between two pushes does not change what it computes.  Argument errors return SSQ_EINVAL and leave the
 * stream as it was; ssq_istream_create checks its arguments before it looks at ctx. */
typedef struct ssq_istream ssq_istream;
ssq_status ssq_istream_create(ssq_ctx* ctx, int64_t channels, int64_t n_frames_total, int64_t n_out,
                              int64_t max_frames, const double* window, int64_t win_n, int n_fft, int hop,
                              int win_exp, int mode, double fs, int out_format, ssq_istream** out);
void ssq_istream_destroy(ssq_istream* s);
int64_t ssq_istream_total_samples(const ssq_istream* s);
int64_t ssq_istream_samples_after(const ssq_istream* s, int64_t n_new);
ssq_status ssq_istream_push(ssq_istream* s, const float* d_Sx, int64_t n_new, float scale, void* d_out,
                            int64_t* samples_written);

/* pinned host memory helpers for the host-buffer path */
ssq_status ssq_host_alloc(void** p, size_t bytes);
void ssq_host_free(void* p);
/* plain cudaMemcpyAsync on a caller-provided cudaStream_t; kind 1 = host to device, 2 = device to host */
ssq_status ssq_memcpy_async(void* dst, const void* src, size_t bytes, int kind, void* cuda_stream);
/* NUMA node of the device's PCIe function (-1: unknown), and pinned host memory placed on it (the host gather of a
 * multi-GPU box should not cross the socket interconnect); falls back to ssq_host_alloc when the node is unknown */
ssq_status ssq_device_numa_node(int device, int* node);
ssq_status ssq_host_alloc_near(void** p, size_t bytes, int device);

#ifdef __cplusplus
}
#endif
#endif /* SSQCUDA_H */

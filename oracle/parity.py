"""Parity gates of SURVEY.md 8(d) -- TEST INFRASTRUCTURE, NOT PRODUCT (tests/, bench.py's parity leg).

north_star: "reassignment bin indices identical except where w falls within fp32 rounding of a bin edge,
with such cases counted and reported".  This module turns that sentence into a decision per (source bin,
frame): given the destination bins the CUDA kernel used (`kb`, written by the kernel itself) and the float64
oracle's Sx, dSx, w and arg-min bins, every mismatch is classified as

  within_edge        the device bin is what the reference's rule (ssq_stft.rs:276-301: nearest grid point,
                     ties to the lower index, clamp) gives for some w' with |w' - w_f64| <= tol, tol < dw/2;
  ill_conditioned    the same with tol >= dw/2: |Sx| is so far below the frame's spectral level that an fp32
                     transform cannot resolve Im(dSx/Sx) to half a bin;
  below_energy_gate  SURVEY 8(d)'s gate: |Sx| < n_fft eps32 max_k|Sx| of the frame -- outside the comparison;
  gate_edge          one side gated the bin (|Sx| < gamma), the other did not, and |Sx| is within the fp32
                     error of gamma;
  unexplained        everything else.  The tests and bench.py assert unexplained == 0.

tol is DERIVED from the fp32 error model of the kernel, not fitted to the mismatches:
  * one packed complex FFT per frame, Z = FFT(x w + i x dw s): each output carries an absolute error of
    about eps32 * sqrt(log2 n_fft) * R, R = rms_k |Z[k]| over the frame (random-walk growth of a
    radix-2^k FFT; Schatzman 1996) -- C_FFT below is the allowance in units of eps32 * R;
  * 2 Sx = Z[k] + conj Z[N-k], 2 V = (Z[k] - conj Z[N-k]) / i inherit it; q = Im(V / Sx) then moves by
    (e / |Sx|) (1 + |V / Sx|), e = C_FFT eps32 R; in grid units that is times cphase = (n_freqs-1)/(pi s);
  * the closed form |k - q cphase| adds a few roundings of its own magnitude (rcp.approx is 1 ulp):
    C_ARITH eps32 (k + |q| cphase).
`emulate_fp32_kernel` restates the kernel's arithmetic in NumPy float32 so the constants can be checked on a
CPU (tests/test_parity_gate_cpu.py): over the input families of the GPU tests (noise, the neural recipe,
tones, tiny amplitudes, random windows) the worst observed |binf32 - binf64| / tol of that restatement
(pocketfft in float32) is 0.09 with C_FFT = 12, C_ARITH = 8.  The CUDA kernels are noisier than pocketfft -- their
twiddles are products of up to 9 table entries (stft_r1024.cuh) and the quotient uses rcp.approx: measured on the
GPU, the worst |w32 - w64| / tol over ~1e6 bins is 0.3 (n_fft 512, noise-like input) to 0.8 (tonal input, where
half a million ill-conditioned bins sample the error distribution far into its tail) -- C_FFT = 12 is about six
standard deviations of the kernels' error, which is what "fp32 rounding" has to mean when every one of 1e7 bins is
held to it.  On well-conditioned bins the bound stays far below a bin (`max_tol_at_edge_flips`, typically 0.005);
every GPU test and bench.py report the ratio for the device's own w (`max_err_over_tol`) and assert it <= 1.
"""
from __future__ import annotations

import math

import numpy as np

from . import ssq_oracle as O

EPS32 = float(np.finfo(np.float32).eps)
C_FFT = 12.0
C_ARITH = 8.0


def s_scale_of(window_fit: np.ndarray) -> float:
    """The kernel packs z = x w + i x dw s with s = sqrt(sum w^2 / sum dw^2) (ssqcuda.cu stft_tables)."""
    dw = O.diff_window(np.asarray(window_fit, dtype=np.float64))
    sd = float((dw * dw).sum())
    sw = float((window_fit * window_fit).sum())
    return math.sqrt(sw / sd) if sd > 0.0 and sw > 0.0 else 1.0


def stft_bin_tolerance(Sx, dSx, n_fft, fs, window_fit):
    """tol [n_freqs, n_frames] in units of the ssq grid step, and the frame levels R [n_frames]."""
    n_freqs = Sx.shape[0]
    s = s_scale_of(window_fit)
    V = dSx * (s / fs)
    p = np.abs(Sx) ** 2 + np.abs(V) ** 2
    full = 2.0 * p.sum(axis=0) - p[0]
    if n_fft % 2 == 0:
        full = full - p[-1]
    R = np.sqrt(np.maximum(full, 0.0) / n_fft)  # rms over the n_fft bins of Z
    cphase = (n_freqs - 1.0) / (math.pi * s)
    aS = np.maximum(np.abs(Sx), 1e-300)
    ratio = np.abs(V) / aS
    with np.errstate(over="ignore", invalid="ignore"):
        tol = C_FFT * EPS32 * cphase * (R[None, :] / aS) * (1.0 + ratio)
        tol = tol + C_ARITH * EPS32 * (np.arange(n_freqs)[:, None] + ratio * cphase)
    return np.nan_to_num(tol, nan=np.inf, posinf=np.inf), R


def classify_stft_bins(kb_dev, aux_o, n_fft, fs, gamma=None, w_dev=None):
    """kb_dev: int [n_freqs, n_frames] from the kernel (-1 gated).  aux_o: the oracle's aux dict
    (Sx, dSx, w, k, window).  w_dev: the kernel's own w (Hz), optional -> max_err_over_tol.
    Returns the report dict."""
    Sx, dSx, w_o, k_o = aux_o["Sx"], aux_o["dSx"], aux_o["w"], aux_o["k"]
    n_freqs, n_frames = Sx.shape
    kb_dev = np.asarray(kb_dev).astype(np.int64)
    assert kb_dev.shape == k_o.shape
    g = 10.0 * O.EPS64 if gamma is None else float(gamma)
    dw = 0.5 * fs / (n_freqs - 1.0)
    tol, R = stft_bin_tolerance(Sx, dSx, n_fft, fs, aux_o["window"])
    mism = kb_dev != k_o
    gated_o, gated_d = k_o < 0, kb_dev < 0
    gate_diff = gated_o ^ gated_d
    # |Sx| against gamma with the fp32 error of Sx itself
    gate_edge = gate_diff & (np.abs(np.abs(Sx) - g) <= C_FFT * EPS32 * R[None, :] + 4 * EPS32 * np.abs(Sx))
    with np.errstate(invalid="ignore", over="ignore"):
        binf = np.where(np.isfinite(w_o), w_o / dw, np.nan)
    # the reference's rule applied to w' in [binf - tol, binf + tol] can give any bin in [lo, hi]:
    # nearest grid point with ties to the lower index = ceil(b - 0.5); clamp to the grid
    with np.errstate(invalid="ignore", over="ignore"):
        lo = np.ceil(np.nan_to_num(binf - tol, nan=0.0, neginf=-1e18) - 0.5)
        hi = np.ceil(np.nan_to_num(binf + tol, nan=0.0, posinf=1e18) - 0.5)
    lo = np.clip(lo, 0, n_freqs - 1)
    hi = np.clip(hi, 0, n_freqs - 1)
    consistent = (kb_dev >= lo) & (kb_dev <= hi) & ~gated_d & ~gated_o
    colmax = np.abs(Sx).max(axis=0, keepdims=True)
    below_gate = np.abs(Sx) < n_fft * EPS32 * np.maximum(colmax, 1e-300)
    well = tol < 0.5
    within_edge = mism & consistent & well & ~below_gate
    ill = mism & consistent & ~well & ~below_gate
    # SURVEY 8(d): bins whose |Sx| lies below n_fft eps32 of the frame's peak are outside the comparison (an fp32
    # transform does not resolve them: for tonal input their error is set by the tone, not by the white-noise model)
    unexplained = mism & ~(consistent | gate_edge | below_gate)
    rep = dict(
        bins_total=int(mism.size), mismatch_total=int(mism.sum()), within_edge=int(within_edge.sum()),
        ill_conditioned=int(ill.sum()), below_energy_gate=int((mism & below_gate).sum()),
        gate_edge=int((mism & gate_edge).sum()), unexplained=int(unexplained.sum()),
        mismatch_above_energy_gate=int((mism & ~below_gate).sum()),
        max_tol_at_edge_flips=float(tol[within_edge].max()) if within_edge.any() else 0.0)
    if w_dev is not None:
        both = np.isfinite(w_o) & np.isfinite(w_dev) & np.isfinite(tol) & (tol > 0)
        with np.errstate(invalid="ignore", over="ignore"):
            ratio = np.abs(np.asarray(w_dev, dtype=np.float64) - w_o) / dw / tol
        sel = both & ~below_gate
        rep["max_err_over_tol"] = float(ratio[sel].max()) if sel.any() else 0.0  # bins above the energy gate
        rep["max_err_over_tol_all_bins"] = float(ratio[both].max()) if both.any() else 0.0
    rep["_unexplained_mask"] = unexplained
    return rep


def public(rep):
    """The report without the mask (JSON-able)."""
    return {k: v for k, v in rep.items() if not k.startswith("_")}


def reaccumulate(Sx_o, kb_dev, fs, squeezing="sum"):
    """Tx the reference's accumulation (ssq_stft.rs:290-299) gives for the ORACLE's Sx with the DEVICE's bins:
    equal to the device's Tx within rtol iff the kernel put every value where it says it did."""
    n_freqs, n_frames = Sx_o.shape
    dw = 0.5 * fs / (n_freqs - 1.0)
    T = np.zeros_like(Sx_o)
    cols = np.arange(n_frames)
    for i in range(n_freqs):
        ok = kb_dev[i] >= 0
        wgt = Sx_o[i] if squeezing != "lebesgue" else np.full(n_frames, 1.0 / n_freqs + 0j)
        np.add.at(T, (kb_dev[i][ok], cols[ok]), wgt[ok] * dw)
    return T


# ---------------------------------------------------------------------------------------------
# NumPy float32 restatement of the kernel's arithmetic (the same formulas, a different FFT
# factorisation): used on the CPU to check the tolerance model and that the gate has teeth.
# ---------------------------------------------------------------------------------------------
def emulate_fp32_kernel(x, window, n_fft, hop, fs, padtype="reflect", gamma=None, rule="reference"):
    """Returns kb [n_freqs, n_frames] (int, -1 gated) and binf (float32) the way the CUDA kernels compute
    them (stft_h32r.cuh h32r_item / stft_r1024.cuh r1k_item), in float32 throughout.
    rule: 'reference' | 'ties_up' | 'floor' | 'drop_out_of_range' -- the wrong rules exist to show that the
    classification rejects them."""
    x = np.asarray(x, dtype=np.float64)
    wfit = O.fit_window(np.asarray(window, dtype=np.float64), n_fft)
    dwin = O.diff_window(wfit)
    s = s_scale_of(wfit)
    padded = O._pad_stft(x, n_fft, padtype).astype(np.float32)
    fr = O._frames(padded, n_fft, hop)
    n_freqs = n_fft // 2 + 1
    z = (fr * wfit.astype(np.float32)[None, :]).astype(np.float32) + 1j * (
        fr * (dwin * s).astype(np.float32)[None, :]).astype(np.float32)
    Z = np.fft.fft(z.astype(np.complex64), axis=1)
    assert Z.dtype == np.complex64
    k = np.arange(n_freqs)
    Zk = Z[:, k]
    Zn = Z[:, (n_fft - k) % n_fft]
    f32 = np.float32
    c = (Zk.real + Zn.real).astype(f32)
    d = (Zk.imag - Zn.imag).astype(f32)
    a = (Zk.imag + Zn.imag).astype(f32)
    b = (Zn.real - Zk.real).astype(f32)
    den = (c * c + d * d).astype(f32)
    num = (b * c - a * d).astype(f32)
    cphase = f32((n_freqs - 1.0) / (math.pi * s))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        q = (num * (f32(1.0) / den)).astype(f32)
        binf = np.abs(k.astype(f32)[None, :] - q * cphase).astype(f32)
        if rule == "ties_up":
            r = np.floor(binf + f32(0.5))
        elif rule == "floor":
            r = np.floor(binf)
        else:
            r = np.ceil(binf - f32(0.5))
    g = 10.0 * O.EPS64 if gamma is None else float(gamma)
    gate2 = f32(-1.0) if g < 0 else f32(min(4.0 * g * g, 3.0e38))
    kb = np.clip(np.nan_to_num(r, nan=0.0, posinf=1e9, neginf=-1e9), 0, n_freqs - 1).astype(np.int64)
    if rule == "drop_out_of_range":
        kb = np.where(np.nan_to_num(r, nan=0.0) > n_freqs - 1, -1, kb)
    kb = np.where(den < gate2, -1, kb)
    return kb.T.copy(), binf.T.copy()


# =============================================================================================
# ssq_cwt (ssq_cwt.rs:116-222): same decision per (scale, time column)
# =============================================================================================
# fp32 error model of the CWT kernels (cwt_kernels.cuh):
#   * x-hat = FFT(padded x) in fp32: absolute error ~ eps32 sqrt(log2 L) * rms_k|x-hat| per bin, which
#     reaches row i as (1/L) ||psi-hat_i||_2 times that (white error through the wavelet filter);
#   * psi-hat is evaluated in fp32 as exp(60 ln w - w^3 - 39.9) (GMW) / exp(-(w-6)^2/2) (Morlet): the exponent,
#     of magnitude up to ~60, carries an absolute rounding of ~60 eps32, i.e. a RELATIVE error of ~4e-6 on
#     psi-hat per spectrum bin, quasi-random in k -- this, not the FFT, dominates: delta W ~ C_PSI eps32 rms|W_i|;
#   * the inverse FFT adds eps32 sqrt(log2 L) rms_n|W_i|.
# e_W[i] = eps32 (C_CWT rms_n|W_i| + C_FFT ||x_pad||_2 ||psi-hat_i||_2 / L), same for dW with psi-hat xi / dt.
# w = |Im(dW / W)| / 2 pi moves by (e_D + |dW/W| e_W) / (2 pi |W|); the bin coordinate is (w - f0) / step or
# (log2 w - f0) / step, rounded half away from zero; bins outside the grid are dropped.
C_CWT = 128.0


def cwt_row_errors(Wx, dWx, x, wavelet, scales, dt, padtype):
    """(e_W, e_D) per row of Wx, dWx: the fp32 error bound of each row (see above)."""
    ns, N = Wx.shape
    L = O.next_power_of_2(N + N // 2)
    padded = O.pad_zero_cwt(x, L) if padtype == "zero" else O.pad_reflect_cwt(np.asarray(x, dtype=np.float64), L)
    xnorm = float(np.sqrt((padded * padded).sum()))
    xi = O.xifn(1.0, L)
    eW = np.empty(ns)
    eD = np.empty(ns)
    for i, s in enumerate(scales):
        ps = O.generate_wavelet_fourier(xi, s, wavelet)
        eW[i] = EPS32 * (C_CWT * np.sqrt((np.abs(Wx[i]) ** 2).mean()) + C_FFT * xnorm * np.sqrt((ps * ps).sum()) / L)
        dps = ps * xi / dt
        eD[i] = EPS32 * (C_CWT * np.sqrt((np.abs(dWx[i]) ** 2).mean()) + C_FFT * xnorm * np.sqrt((dps * dps).sum()) / L)
    # the kernel evaluates psi-hat as exactly 0 below ~2e-18 (GMW: w outside (1, 4.5)) / 2e-16 (Morlet: w > 14.5) of
    # its peak (cwt_kernels.cuh psihat); the dropped tail is at most floor * sum_k |x-hat_k| / L in W
    xh1 = float(np.abs(np.fft.fft(padded)).sum()) / L
    floor_rel, peak = (2.2e-16, 1.0622519320271968) if wavelet == "morlet" else (2.0e-18, 2.0 * math.exp(39.914641217580179))
    return eW + floor_rel * peak * xh1, eD + floor_rel * peak * xh1 * (math.pi / dt)


def cwt_bin_tolerance(aux_o, x, wavelet, dt, padtype, ssq_freqs, row_err=None):
    """row_err: (e_W, e_D) of the rows, when aux_o holds a slice of columns of them (`cwt_row_errors` needs whole
    rows)."""
    Wx, dWx, w_o, scales = aux_o["Wx"], aux_o["dWx"], aux_o["w"], aux_o["scales"]
    eW, eD = row_err if row_err is not None else cwt_row_errors(Wx, dWx, x, wavelet, scales, dt, padtype)
    aW = np.abs(Wx)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        # delta(dW / W) <= (e_D + |dW / W| e_W) / (|W| - e_W): unbounded once |W| is within the error itself
        den = aW - 2.0 * eW[:, None]
        dw_abs = np.where(den > 0, (eD[:, None] + (np.abs(dWx) / np.maximum(aW, 1e-300)) * eW[:, None])
                          / (2.0 * math.pi * np.maximum(den, 1e-300)), np.inf)
        dw_abs = dw_abs + C_ARITH * EPS32 * np.where(np.isfinite(w_o), w_o, 0.0)
    nf = len(ssq_freqs)
    is_log = (ssq_freqs[1] / ssq_freqs[0] > 1.1) if nf > 1 else False
    return np.nan_to_num(dw_abs, nan=np.inf, posinf=np.inf), is_log, eW


def classify_cwt_bins(kb_dev, aux_o, x, wavelet, dt, padtype, ssq_freqs, flipud=True, gamma=None, w_dev=None,
                      row_err=None):
    """kb_dev: int [ns, N]: destination ROW of Tx for every (scale, column), -1 where nothing was added (gated,
    non-finite w, out of range).  aux_o: oracle aux (Wx, dWx, w, k, scales), or a slice of its columns with
    row_err = (e_W, e_D) of the whole rows (`cwt_row_errors`)."""
    Wx, w_o, k_o = aux_o["Wx"], aux_o["w"], aux_o["k"]
    ns, N = Wx.shape
    nf = len(ssq_freqs)
    kb_dev = np.asarray(kb_dev).astype(np.int64)
    assert kb_dev.shape == k_o.shape
    g = 10.0 * O.EPS64 if gamma is None else float(gamma)
    dw_abs, is_log, eW = cwt_bin_tolerance(aux_o, x, wavelet, dt, padtype, ssq_freqs, row_err)
    if is_log:
        f0 = math.log2(ssq_freqs[0])
        step = (math.log2(ssq_freqs[nf - 1]) - f0) / (nf - 1.0) if nf > 1 else 1.0
        coord = lambda w: (np.log2(w) - f0) / step
    else:
        f0 = ssq_freqs[0]
        step = (ssq_freqs[nf - 1] - f0) / (nf - 1.0) if nf > 1 else 1.0
        coord = lambda w: (w - f0) / step
    fin = np.isfinite(w_o)
    with np.errstate(all="ignore"):
        wlo = np.where(fin, np.maximum(w_o - dw_abs, 0.0), np.nan)
        whi = np.where(fin, w_o + dw_abs, np.nan)
        clo, chi, c0 = coord(wlo), coord(whi), coord(np.where(fin, w_o, np.nan))
        if step < 0:
            clo, chi = chi, clo
        tol = np.maximum(np.abs(chi - c0), np.abs(c0 - clo))  # in grid units (asymmetric for the log grid)
        # round half away from zero over [clo, chi]; the set of reachable bins is an interval
        rlo = np.sign(clo) * np.floor(np.abs(clo) + 0.5)
        rhi = np.sign(chi) * np.floor(np.abs(chi) + 0.5)
    rlo = np.nan_to_num(rlo, nan=-1e18, neginf=-1e18, posinf=1e18)
    rhi = np.nan_to_num(rhi, nan=1e18, neginf=-1e18, posinf=1e18)
    bin_dev = np.where(kb_dev >= 0, (nf - 1 - kb_dev) if flipud else kb_dev, -1)
    added_d, added_o = kb_dev >= 0, k_o >= 0
    mism = kb_dev != k_o
    # device added at bin b: b must be reachable; device dropped: some reachable bin must lie outside the grid, or the
    # gate |W| < gamma is within the fp32 error of W
    reachable = added_d & (bin_dev >= rlo) & (bin_dev <= rhi)
    drop_ok = ~added_d & ((rlo < 0) | (rhi > nf - 1) | ~fin)
    gate_edge = (added_d ^ added_o) & (np.abs(np.abs(Wx) - g) <= eW[:, None] + 4 * EPS32 * np.abs(Wx))
    unresolved = ~np.isfinite(dw_abs)  # |W| within the fp32 error of W itself: any outcome (bin or drop) is reachable
    consistent = reachable | drop_ok | gate_edge | unresolved
    tol = np.nan_to_num(tol, nan=np.inf, posinf=np.inf)
    well = tol < 0.5
    unexplained = mism & ~consistent
    rep = dict(bins_total=int(mism.size), mismatch_total=int(mism.sum()),
               within_edge=int((mism & consistent & well & ~gate_edge).sum()),
               ill_conditioned=int((mism & consistent & ~well & ~gate_edge).sum()),
               gate_edge=int((mism & gate_edge).sum()), unexplained=int(unexplained.sum()),
               is_log=bool(is_log))
    if w_dev is not None:
        w_dev = np.asarray(w_dev, dtype=np.float64)
        both = fin & np.isfinite(w_dev) & np.isfinite(dw_abs) & (dw_abs > 0)
        with np.errstate(all="ignore"):
            ratio = np.abs(w_dev - w_o) / dw_abs
        rep["max_err_over_tol"] = float(ratio[both].max()) if both.any() else 0.0
    rep["_unexplained_mask"] = unexplained
    return rep


def reaccumulate_cwt(Wx_o, kb_dev, n_rows, squeezing="sum"):
    """ssq_cwt.rs:192-207 with the DEVICE's destination rows: Tx[k, j] += Wx[i, j] (or 1/n_scales)."""
    ns, N = Wx_o.shape
    T = np.zeros((n_rows, N), dtype=np.complex128)
    cols = np.arange(N)
    for i in range(ns):
        ok = kb_dev[i] >= 0
        wgt = Wx_o[i] if squeezing != "lebesgue" else np.full(N, 1.0 / ns + 0j)
        np.add.at(T, (kb_dev[i][ok], cols[ok]), wgt[ok])
    return T


def emulate_fp32_cwt_kernel(x, wavelet, scales, dt, padtype, ssq_freqs, flipud=True, gamma=None):
    """NumPy float32 restatement of cwt_kernels.cuh (peak-normalised GMW, fp32 psi-hat, complex64 FFTs, the
    reassignment arithmetic of ssq_cwt_reassign_kernel).  Returns kb [ns, N] and w (float32, Hz)."""
    f32 = np.float32
    x = np.asarray(x, dtype=np.float64)
    N = len(x)
    L = O.next_power_of_2(N + N // 2)
    padded = (O.pad_zero_cwt(x, L) if padtype == "zero" else O.pad_reflect_cwt(x, L)).astype(f32)
    xh = np.fft.fft(padded.astype(np.complex64))
    idx = np.arange(L)
    xi = (f32(6.283185307179586) * idx.astype(f32) / f32(L)).astype(f32)
    half = idx <= L // 2
    ns = len(scales)
    nf = len(ssq_freqs)
    n1 = (L - N) // 2
    K = 1.0 if wavelet == "morlet" else 2.0 * math.exp(39.914641217580179)
    g = 10.0 * O.EPS64 if gamma is None else float(gamma)
    is_log = (ssq_freqs[1] / ssq_freqs[0] > 1.1) if nf > 1 else False
    if is_log:
        f0 = math.log2(ssq_freqs[0]); inv_step = (nf - 1.0) / (math.log2(ssq_freqs[nf - 1]) - f0) if nf > 1 else 1.0
    else:
        f0 = ssq_freqs[0]; inv_step = (nf - 1.0) / (ssq_freqs[nf - 1] - f0) if nf > 1 else 1.0
    kb = np.full((ns, N), -1, dtype=np.int64)
    wout = np.full((ns, N), np.inf, dtype=np.float32)
    for i, s in enumerate(scales):
        w = (f32(s) * xi).astype(f32)
        ps = np.zeros(L, dtype=f32)
        with np.errstate(all="ignore"):
            if wavelet == "morlet":
                ok = half & (w >= 0) & (w <= 14.5)
                d = (w - f32(6.0)).astype(f32)
                v = f32(1.0622519320271968) * (np.exp(f32(-0.5) * d * d) - f32(1.5229979744712629e-08) * np.exp(f32(-0.5) * w * w))
            else:
                ok = half & (w >= 1.0) & (w <= 4.5)
                v = np.exp(f32(60.0) * np.log(w) - w * w * w - f32(39.914641217580179))
        ps[ok] = v.astype(f32)[ok]
        Y = (xh * ps).astype(np.complex64)
        W = (np.fft.ifft(Y) ).astype(np.complex64)[n1:n1 + N]
        D = (np.fft.ifft((Y * (1j * (xi * f32(1.0 / dt)))).astype(np.complex64))).astype(np.complex64)[n1:n1 + N]
        c, d_, a, b = W.real.astype(f32), W.imag.astype(f32), D.real.astype(f32), D.imag.astype(f32)
        mag = np.hypot(c, d_)
        with np.errstate(all="ignore"):
            ww = np.abs((b * c - a * d_) / ((c * c + d_ * d_) * f32(6.283185307179586))).astype(f32)
            vv = ((np.log2(ww) - f32(f0)) * f32(inv_step)) if is_log else ((ww - f32(f0)) * f32(inv_step))
            r = np.sign(vv) * np.floor(np.abs(vv) + f32(0.5))
        ok = (mag >= f32(g / K)) & np.isfinite(ww) & np.isfinite(r) & (r >= 0) & (r < nf)
        bins = np.where(ok, r, 0).astype(np.int64)
        kb[i] = np.where(ok, (nf - 1 - bins) if flipud else bins, -1)
        wout[i] = np.where(mag >= f32(g / K), ww, np.inf)
    return kb, wout

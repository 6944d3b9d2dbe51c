"""Every plan of the row-FFT engine (`fft_plan` / `fft_plan_rows` / `fft_run`, cwt_host.inl and stft_rows.inl), from
rows of 4 points to rows of 2^27, against a float64 oracle that holds each output ROW to its own magnitude.

The CWT, the STFT rows path (n_fft above 4096 and every n_fft that is not a power of two, forward and inverse) and the
two-integral icwt all run on one Stockham engine whose pass sequence depends only on log2 of the row length, and a CWT
row may enter it at up to three points (`cwt_skip_level`: leading passes that are pure broadcasts for band-limited
rows are not launched).  The other parity tests compare with `max|a - b| / max|b|` over a whole array; a large-scale
CWT row is a few hundred times smaller than the array maximum, so a pass that is wrong only on those rows (the ones
that take the skip entry points) could be wrong by percents unseen.  Here each row r -- one CWT row, one STFT frame,
one inverse -- must satisfy

    ||dev_r - ref_r||_2 <= B_L2 ||ref_r||_2   and   max |dev_r - ref_r| <= B_MAX max |ref_r|

(`test_per_row_check_catches_what_the_array_maximum_misses` shows the difference on an oracle map).

Without a GPU: the planners restated (constants read from the source), the invariants the kernels rely on, the case
table with proof that it reaches every (plan, entry point, skip level, fused / stand-alone) cell, and a per-row
float64 oracle on scipy.fft (workers) pinned to `O.cwt`, `O.stft`, `O.istft` and `O.icwt`.

On the GPU, each case asserts the kernel it reached:
* cwt (W, dW) and ssq_cwt (fused where `cwt_fused_ok` holds, stand-alone everywhere; every bin classified, Tx per Tx
  row against the oracle's W accumulated over the device's bins) for every log2 L from 2 to 27 at the smallest and
  the largest N of its range, scales 2, N/2 and each skip threshold x (1 -+ 2^-12).  From log2 L = 24 on, the bins are
  classified on column slices of 2^16 at the start, middle and end, and one wavelet is run per N (GMW on the smallest,
  Morlet on the largest); the per-row W, dW checks stay whole-row.  The options (l2 norm, zero padding, rpadded) on
  one size per pass count; 3 channels at L = 2^27, where the passes take 2 rows per launch; the fused / stand-alone
  switch at ns N = 2^31.
* the STFT rows path on every plan its frames reach: powers of two 2^11 .. 2^15 and one odd (Bluestein) n_fft per row
  length 2^7 .. 2^17, stft per frame (2 channels through `Engine`), ssq_stft (every bin classified up to n_fft 2^14:
  the oracle's arg-min is quadratic in n_fft; above, Sx, dSx per frame and w where |Sx| carries the frame), and istft
  against the oracle.  One tile of the rows-mode kernels holds at least one frame in shared memory, so frames are
  limited to 45 509 points forward and 51 197 inverse; longer ones are refused with the limit in the message.  The
  plans of longer rows are fft_plan's, run by the CWT and the icwt cases.
* the two-integral icwt at x_len = 2^k, k = 2 .. 27, and at one Bluestein length per row length 2^3 .. 2^27.

Host cost: the per-row oracle is one scipy transform per row (about 3 s at 2^27 with 8 workers); the Bluestein
tables of the library are a double-precision DFT on the host (seconds and about 2 GiB at rows of 2^27, the icwt case).
Rows whose band holds no energy (N = 2, whose reflect padding is periodic with period 2) are held to the bound of what
the kernel drops below its psi-hat cut-off instead of their own size.
"""
import gc
import math
import os
import re

import numpy as np
import pytest
import scipy.fft as sfft

from oracle import parity as P
from oracle import ssq_oracle as O

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "ssqueeze_rs_b200", "csrc")
WORKERS = max(1, min(8, os.cpu_count() or 1))
EPS32 = float(np.finfo(np.float32).eps)
GAMMA = 10.0 * O.EPS64


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


CWT_HOST, ROWS_HOST, CWT_KERNELS = _src("cwt_host.inl"), _src("stft_rows.inl"), _src("cwt_kernels.cuh")


def _re(pattern, text):
    m = re.search(pattern, text)
    assert m, "source moved: " + pattern
    return m.groups()


# ---------------------------------------------------------------------------------------------------------------------
# the planners, restated (constants read from the source)
# ---------------------------------------------------------------------------------------------------------------------
# cwt_skip_level (cwt_host.inl): B = wmax L / (2 pi scale) (1 + MARGIN) + PLUS; wmax 14.5 Morlet, 4.5 GMW
WMAX_MORLET, WMAX_GMW = map(float, _re(r"wmax = \(c\.wavelet == SSQ_WAVELET_MORLET\) \? ([0-9.]+) : ([0-9.]+);",
                                       CWT_HOST))
MARGIN, PLUS = map(float, _re(r"B = wmax \* L / \(2\.0 \* SSQ_PI \* scale\) \* \(1\.0 \+ ([0-9.e+-]+)\) \+ ([0-9.]+);",
                              CWT_HOST))
WMAX = {"gmw": WMAX_GMW, "morlet": WMAX_MORLET}
# cwt_fused_ok (cwt_host.inl): last radix 7, log2L - 7 >= 5, log2L >= 12, pitch < 2^30, ns pitch < 2^31
FUSED_NS_MIN, FUSED_L2_MIN, FUSED_PITCH_SHIFT, FUSED_ELEM_SHIFT = map(int, _re(
    r"pl\.log2L - 7 >= (\d+) && pl\.log2L >= (\d+) && pitch < \(\(int64_t\)1 << (\d+)\) &&\s*"
    r"ns \* pitch < \(\(int64_t\)1 << (\d+)\);", CWT_HOST))
# fft_plan (cwt_host.inl): one pass up to 2^12; 7, middle, 7 from 2^18; 7,7 at 2^14
(ONE_PASS_MAX,) = map(int, _re(r"if \(log2L <= (\d+)\) \{\s*p\.npass = 1;", CWT_HOST))
(OUTER7_MIN,) = map(int, _re(r"if \(log2L >= (\d+)\) \{\s*const int rem = log2L - 14;", CWT_HOST))
# fft_plan_rows (stft_rows.inl): 7, l2 - 7 for rows of 2^11 / 2^12
ROWS_SPECIAL = tuple(map(int, _re(r"if \(l2 != (\d+) && l2 != (\d+)\) return fft_plan\(l2\);", ROWS_HOST)))
(MAX_L2,) = map(int, _re(r"if \(l2 > (\d+)\) return ssq_fail\(ctx, SSQ_EUNSUPPORTED, \"cwt: padded length", CWT_HOST))
PAD_RULE = _re(r"const int64_t L = ssqhost::next_power_of_2\((c\.n \+ c\.n / 2)\);", CWT_HOST)
T32_MIN_L2 = int(_re(r"log2T == 5 plans have L >= 2\^(\d+)", CWT_HOST)[0])
# the rows-mode tile kernels (stft_rows.inl): a tile holds at least one frame of (n_freqs | 1) complex64, plus one
# byte tag per frequency for each warp of the forward kernel, in a shared-memory budget of ROWS_SMEM bytes
ROWS_SMEM = int(_re(r"const size_t budget = std::min<size_t>\(\(size_t\)ctx->max_smem_optin, (\d+) \* 1024\);",
                    ROWS_HOST)[0]) * 1024


def fft_plan(l2):
    """fft_plan (cwt_host.inl) -> (radices, log2T)."""
    if l2 <= ONE_PASS_MAX:
        return [l2], 0
    if l2 >= OUTER7_MIN:
        rem = l2 - 14
        if rem == 7:
            mid = [7]
        elif rem <= 7:
            mid = [rem]
        elif rem >= 11:
            mid = [7, rem - 7]
        else:
            mid = [(rem + 1) // 2, rem // 2]
        return [7] + mid + [7], 5
    if l2 == 14:
        return [7, 7], 5
    n7, rem = l2 // 7, l2 - 7 * (l2 // 7)
    if rem >= 4:
        return [7] * n7 + [rem], 5
    two = 7 + rem
    return [7] * (n7 - 1) + [(two + 1) // 2, two // 2], 5


def fft_plan_rows(l2):
    """fft_plan_rows (stft_rows.inl)."""
    if l2 not in ROWS_SPECIAL:
        return fft_plan(l2)
    return [7, l2 - 7], 5


def rows_tile_smem(n_freqs, F, nw, fwd):
    """rows_tile_smem (stft_rows.inl)."""
    acc = F * (n_freqs | 1) * 8
    return acc + nw * ((n_freqs + 7) & ~7) if fwd else acc


def rows_max_nfft(fwd):
    """The largest n_fft whose one-frame tile fits ROWS_SMEM (rows_max_nfft, stft_rows.inl)."""
    m = ROWS_SMEM // (9 if fwd else 8) + 2
    while m > 1 and rows_tile_smem(m, 1, 1, fwd) > ROWS_SMEM:
        m -= 1
    return 2 * m - 1


def pad_len(n):
    """next_power_of_2(n + n / 2) (cwt_prepare, cwt_host.inl; host_math.h)."""
    m = n + n // 2
    return 1 << max(0, (m - 1).bit_length())


def n_range(l2):
    """(smallest, largest) N whose padded CWT length is 2^l2."""
    def top(L):  # largest n with n + n // 2 <= L
        n = (2 * L) // 3 + 2
        while n + n // 2 > L:
            n -= 1
        return n
    return top(1 << (l2 - 1)) + 1, top(1 << l2)


def skip_level(l2, wavelet, scale):
    """cwt_skip_level (cwt_host.inl) for the plan of 2^l2 and a scale (the double the host sees)."""
    rad, log2T = fft_plan(l2)
    if len(rad) < 2 or log2T != 5 or not scale > 0.0:
        return 0
    L = float(1 << l2)
    B = WMAX[wavelet] * L / (2.0 * math.pi * scale) * (1.0 + MARGIN) + PLUS
    lvl = 1 if B <= L / (1 << rad[0]) else 0
    if lvl == 1 and len(rad) >= 3 and B <= L / (1 << (rad[0] + rad[1])):
        lvl = 2
    return lvl


def levels(l2):
    """Skip levels the plan of 2^l2 admits."""
    rad, log2T = fft_plan(l2)
    if len(rad) < 2 or log2T != 5:
        return [0]
    return [0, 1, 2] if len(rad) >= 3 else [0, 1]


def fused_ok(l2, pitch, ns):
    """cwt_fused_ok (cwt_host.inl), option no_cwt_fused off."""
    rad, log2T = fft_plan(l2)
    if len(rad) < 2 or log2T != 5:
        return False
    return (rad[-1] == 7 and l2 - 7 >= FUSED_NS_MIN and l2 >= FUSED_L2_MIN and pitch < (1 << FUSED_PITCH_SHIFT)
            and ns * pitch < (1 << FUSED_ELEM_SHIFT))


def f32(v):
    return np.asarray(v, dtype=np.float32).astype(np.float64)


def threshold(l2, wavelet, lvl):
    """The scale above which rows of 2^l2 points skip `lvl` passes (B <= L / 2^(bits of the skipped passes))."""
    rad, _ = fft_plan(l2)
    L = float(1 << l2)
    return WMAX[wavelet] * L * (1.0 + MARGIN) / (2.0 * math.pi * (L / (1 << sum(rad[:lvl])) - PLUS))


def case_scales(l2, N, wavelet):
    """Scales 2, N/2 and each skip threshold x (1 -+ 2^-12), exact in fp32, ascending."""
    s = [2.0, N / 2.0]
    for lvl in levels(l2)[1:]:
        t = threshold(l2, wavelet, lvl)
        s += [t * (1 - 2.0 ** -12), t * (1 + 2.0 ** -12)]
    return np.unique(f32(s))


# ---------------------------------------------------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------------------------------------------------
SLICE_FROM_L2 = 24  # classify bins on column slices from here on (host memory)
CWT_CASES = []
for _l2 in range(2, MAX_L2 + 1):
    _lo, _hi = n_range(_l2)
    CWT_CASES.append((_l2, _lo, ("gmw", "morlet") if _l2 < SLICE_FROM_L2 else ("gmw",)))
    CWT_CASES.append((_l2, _hi, ("gmw", "morlet") if _l2 < SLICE_FROM_L2 else ("morlet",)))
CWT_OPTION_CASES = [10, 14, 19, 22]  # 1, 2, 3 and 4 passes
# the rows path takes frames up to ROWS_FWD_MAX points forward and ROWS_INV_MAX inverse (one frame per tile in
# shared memory): powers of two up to 2^15, Bluestein rows up to 2^17; longer frames are refused (ROWS_REFUSED), and
# the plans of longer rows are the CWT / icwt plans (fft_plan_rows = fft_plan from 2^13 on)
ROWS_FWD_MAX, ROWS_INV_MAX = rows_max_nfft(True), rows_max_nfft(False)
ROWS_POW2 = [1 << k for k in range(11, MAX_L2 + 1) if 1 << k <= ROWS_FWD_MAX]
ROWS_BLUE = [min(((3 << k) // 8) | 1, ROWS_FWD_MAX) for k in range(7, 18)]  # odd, in (M/4, M/2] for M = 2^k
ROWS_REFUSED = [1 << 16, ((3 << 17) // 8) | 1, 1 << 20]
ICWT2_LENS = [1 << k for k in range(2, MAX_L2 + 1)] + [((3 << k) // 8) | 1 for k in range(3, MAX_L2 + 1)]
CLASSIFY_STFT_MAX = 1 << 14
BOUNDARY_N, BOUNDARY_NS = 1 << 22, 513  # ns N just above 2^31: the stand-alone path


def rows_M(n_fft):
    pow2 = n_fft & (n_fft - 1) == 0
    M = 1
    while M < (n_fft if pow2 else 2 * n_fft - 1):
        M <<= 1
    return M


def _ids(cases):
    return [f"L2^{l2}-N{N}-{'+'.join(w)}" for l2, N, w in cases]


# ---------------------------------------------------------------------------------------------------------------------
# per-row float64 oracle (restates O._cwt_core, O.stft, O.istft, O.icwt one row at a time on scipy.fft)
# ---------------------------------------------------------------------------------------------------------------------
def cwt_rows(x, wavelet, scales, dt=1.0, padtype="reflect", derivative=True, rpadded=False, l1_norm=True,
             errors=False):
    """Yields (W_r, dW_r | None, err | None) per scale: O.cwt's rows (O._cwt_core), and with `errors`
    err = (e_W, e_D, t_W, t_D): the fp32 bounds of oracle/parity.py's `cwt_row_errors` for the row, and the part of
    them that bounds what the kernel drops below its psi-hat cut-off (t)."""
    x = np.asarray(x, dtype=np.float64)
    N = len(x)
    L = O.next_power_of_2(N + N // 2)
    padded = O.pad_zero_cwt(x, L) if padtype == "zero" else O.pad_reflect_cwt(x, L)
    xh = sfft.fft(padded, workers=WORKERS)
    xi = O.xifn(1.0, L)
    n1 = (L - N) // 2
    sl = slice(0, L) if rpadded else slice(n1, n1 + N)
    if errors:
        xnorm = float(np.sqrt((padded * padded).sum()))
        xh1 = float(np.abs(xh).sum()) / L
        floor_rel, peak = ((2.2e-16, 1.0622519320271968) if wavelet == "morlet"
                           else (2.0e-18, 2.0 * math.exp(39.914641217580179)))
    del padded
    for s in scales:
        ps = O.generate_wavelet_fourier(xi, s, wavelet)
        f = 1.0 if l1_norm else math.sqrt(s)
        W = sfft.ifft(xh * ps, workers=WORKERS)[sl]
        dW = sfft.ifft(xh * (ps * (1j * (xi / dt))), workers=WORKERS)[sl] if derivative else None
        err = None
        if errors:
            tail = floor_rel * peak * xh1
            eW = EPS32 * (P.C_CWT * np.sqrt((np.abs(W) ** 2).mean()) + P.C_FFT * xnorm * np.sqrt((ps * ps).sum()) / L)
            dps = ps * xi / dt
            eD = EPS32 * (P.C_CWT * np.sqrt((np.abs(dW) ** 2).mean()) + P.C_FFT * xnorm * np.sqrt((dps * dps).sum()) / L)
            err = (eW + tail, eD + tail * (math.pi / dt), tail, tail * (math.pi / dt))
            del dps
        del ps
        yield (W * f if f != 1.0 else W), (dW * f if (dW is not None and f != 1.0) else dW), err


def stft_frames(x, n_fft, hop, window, padtype="reflect", frames=None, scale=1.0):
    """O.stft's columns (rfft of each windowed frame of the crate framing) -> [n_fft // 2 + 1, n_frames]."""
    x = np.asarray(x, dtype=np.float64)
    padded = O._pad_stft(x, n_fft, padtype)
    nfr = (len(padded) - n_fft) // hop + 1
    frames = range(nfr) if frames is None else frames
    w = np.asarray(window, dtype=np.float64)[:n_fft] * scale
    out = np.empty((n_fft // 2 + 1, len(frames)), dtype=np.complex128)
    for j, f in enumerate(frames):
        out[:, j] = sfft.rfft(padded[f * hop:f * hop + n_fft] * w, workers=WORKERS)
    return out


def diff_window(w):
    """O.diff_window on scipy.fft."""
    n = len(w)
    k = np.arange(n, dtype=np.float64)
    k[n // 2 + 1:] -= n
    xi = k * (2.0 * math.pi / n)
    Wf = sfft.fft(w, workers=WORKERS)
    Wf = (-Wf.imag * xi) + 1j * (Wf.real * xi)
    return (sfft.ifft(Wf, workers=WORKERS) * n).real * (1.0 / n)


def istft_ref(Sx, window, n_fft, hop, N):
    """O.istft (crate framing, win_exp 1) on scipy.fft."""
    left = O.pad_left(n_fft)
    wsz = O.fit_window(window, n_fft)
    nfr = Sx.shape[1]
    L = N + n_fft - 1
    xr = np.zeros(L)
    for j in range(nfr):
        s = j * hop
        if s + n_fft > L:
            break
        xr[s:s + n_fft] += sfft.irfft(Sx[:, j], n=n_fft, workers=WORKERS) * wsz
    wn = np.zeros(L)
    wpow = wsz ** 2
    for j in range((L - n_fft) // hop + 1):
        wn[j * hop:j * hop + n_fft] += wpow
    nz = wn > np.finfo(np.float64).tiny
    xr[nz] /= wn[nz]
    return xr[left:left + N]


def icwt2_ref(Wx, wavelet, scales, x_len, x_mean=0.0):
    """O.icwt(one_int=False, l1_norm=True) on scipy.fft."""
    xi = O.xifn(1.0, x_len)
    x = np.zeros(x_len)
    for i, s in enumerate(scales):
        ps = O.generate_wavelet_fourier(xi, s, wavelet)
        tmp = sfft.ifft(sfft.fft(Wx[i, :x_len], workers=WORKERS) * ps, workers=WORKERS) * x_len
        x += tmp.real * (1.0 / x_len) * (1.0 / s)
    dj = math.log(scales[1] / scales[0]) if (len(scales) > 1 and scales[1] > scales[0]) else 0.1
    adm = 0.776 if wavelet == "morlet" else 1.0  # cwt.rs:579-583
    return x * ((2.0 / adm) * dj) + x_mean


def broadband(n, seed, scale=3.0):
    """White noise plus a chirp sweeping 0 .. Nyquist, exact in fp32: every CWT row and STFT frame has energy in its
    own band."""
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64) / max(n, 1)
    x = rng.standard_normal(n) * scale + scale * np.sin(np.pi * 0.5 * n * t * t)
    return f32(x)


# ---------------------------------------------------------------------------------------------------------------------
# the per-row criterion
# ---------------------------------------------------------------------------------------------------------------------
# Bounds per family: at least 4x the worst ratio a B200 measured (printed at the end of the GPU run), at most
# 1e-5 (L2) and 1e-4 (max) -- DESIGN §6 / §6b.
B_L2 = 1e-5
B_MAX = 1e-4
# families with their own bounds (DESIGN §6b): the CWT rows and the two-integral icwt carry the fp32 evaluation of
# psi-hat (GMW: 3e-6 rms, 1.3e-5 at most of its value), not only the FFT's rounding; the STFT families are tighter than
# the ceilings; Tx is a max-only bound per element (`_classify_slices`)
BOUNDS = {"cwt W": (3e-5, 5e-5), "cwt dW": (3e-5, 5e-5), "icwt2": (2e-5, 2e-5), "icwt2 bluestein": (2e-5, 2e-5),
          "ssq_cwt Tx": (None, 1e-4)}
for _f in ("stft", "istft", "ssq_stft Sx", "ssq_stft dSx"):
    for _k in ("rows", "bluestein"):
        BOUNDS[f"{_f} {_k}"] = (2e-6, 4e-6)
WORST = {}


def row_ratios(dev, ref):
    dev = np.asarray(dev).astype(np.complex128 if np.iscomplexobj(dev) or np.iscomplexobj(ref) else np.float64)
    ref = np.asarray(ref)
    e = dev - ref
    nr, mr = float(np.linalg.norm(ref)), float(np.abs(ref).max())
    if nr == 0.0:
        return (0.0 if not e.any() else math.inf), (0.0 if not e.any() else math.inf)
    return float(np.linalg.norm(e)) / nr, float(np.abs(e).max()) / mr


def check_row(family, dev, ref, what="", floor=0.0):
    """floor: what the kernel may drop below its psi-hat cut-off; a row entirely below it (no energy in its band: the
    reference is the oracle's tail of psi-hat) is held to the floor instead of its own size."""
    if floor > 0.0 and float(np.abs(ref).max()) <= floor:
        assert float(np.abs(np.asarray(dev) - ref).max()) <= floor, (family, what, "row below the psi-hat cut-off")
        return
    l2, mx = row_ratios(dev, ref)
    w = WORST.setdefault(family, [0.0, 0.0, ""])
    if l2 > w[0]:
        w[0], w[2] = l2, what
    w[1] = max(w[1], mx)
    bl2, bmax = BOUNDS.get(family, (B_L2, B_MAX))
    assert l2 <= bl2 and mx <= bmax, (family, what, l2, mx)


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if WORST:
        print("\nper-row worst ratios (family: L2, max, row of the L2 worst):")
        for k in sorted(WORST):
            print(f"  {k}: {WORST[k][0]:.3e} {WORST[k][1]:.3e} {WORST[k][2]}")


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_restated_planners_read_the_source_constants():
    assert (WMAX_GMW, WMAX_MORLET, MARGIN, PLUS) == (4.5, 14.5, 1e-4, 2.0)
    assert (FUSED_NS_MIN, FUSED_L2_MIN, FUSED_PITCH_SHIFT, FUSED_ELEM_SHIFT) == (5, 12, 30, 31)
    assert (ONE_PASS_MAX, OUTER7_MIN, ROWS_SPECIAL, MAX_L2, T32_MIN_L2) == (12, 18, (11, 12), 27, 11)
    assert PAD_RULE == ("c.n + c.n / 2",)
    # the kernel's psi-hat cut-offs are the host's wmax (cwt_kernels.cuh psihat and the generation early-out)
    assert f"if (w > {WMAX_MORLET}f) return 0.f;" in CWT_KERNELS
    assert f"if (w < 1.0f || w > {WMAX_GMW}f) return 0.f;" in CWT_KERNELS
    assert f"? {WMAX_MORLET}f : {WMAX_GMW}f;" in CWT_KERNELS
    # the other planners that take fft_plan: rows path and icwt both stop at 2^27
    assert "if (l2 > 27) return ssq_fail(ctx, SSQ_EUNSUPPORTED, \"icwt: rows" in CWT_HOST
    assert ROWS_HOST.count("if (l2 > 27) return ssq_fail(ctx, SSQ_EUNSUPPORTED, \"n_fft=%d") == 2
    # the table of the plans
    want = {13: [7, 6], 14: [7, 7], 15: [7, 4, 4], 16: [7, 5, 4], 17: [7, 5, 5], 18: [7, 4, 7], 19: [7, 5, 7],
            20: [7, 6, 7], 21: [7, 7, 7], 22: [7, 4, 4, 7], 23: [7, 5, 4, 7], 24: [7, 5, 5, 7], 25: [7, 7, 4, 7],
            26: [7, 7, 5, 7], 27: [7, 7, 6, 7]}
    for l2 in range(2, 28):
        assert fft_plan(l2) == ((want[l2], 5) if l2 in want else ([l2], 0)), l2
    assert fft_plan_rows(11) == ([7, 4], 5) and fft_plan_rows(12) == ([7, 5], 5)
    # pad rule against the oracle's float-log2 restatement at every range edge
    for l2 in range(2, 28):
        lo, hi = n_range(l2)
        for n in (lo, hi):
            assert pad_len(n) == O.next_power_of_2(n + n // 2) == 1 << l2, (l2, n)
        assert pad_len(hi + 1) == 1 << (l2 + 1) and (l2 == 2 or pad_len(lo - 1) == 1 << (l2 - 1))
    assert n_range(2) == (2, 3) and n_range(12)[1] == 2731 and n_range(22) == (1398102, 2796203)
    assert n_range(27) == (44739244, 89478485)


@pytest.mark.parametrize("planner", ["cwt", "rows"])
def test_plan_invariants(planner):
    plan = fft_plan if planner == "cwt" else fft_plan_rows
    for l2 in range(2 if planner == "cwt" else 7, MAX_L2 + 1):
        rad, log2T = plan(l2)
        assert sum(rad) == l2, (l2, rad)
        # multi-pass plans: radices <= 7 in T = 32 columns; one pass: the whole row of <= 2^12 points, T = 1
        # (fft_pass_kernel, 2 R T complex64 of shared memory)
        assert all(1 <= r <= 7 for r in rad) if len(rad) > 1 else (rad[0] <= ONE_PASS_MAX and log2T == 0), (l2, rad)
        if log2T == 5:
            assert l2 >= T32_MIN_L2, l2
        # grids: the generic pass takes L / (R T) CTAs; a 7-bit pass runs in fft128_pass_kernel (it needs Ns = 1 or
        # Ns >= 32) with L / (128 TC) CTAs, TC = 16 columns, 32 under the fused tail (fft_run)
        bits = 0
        for r in rad:
            if r == 7 and log2T == 5:
                assert bits == 0 or bits >= 5, (l2, rad)
                assert (1 << l2) % (128 * (32 if fused_ok(l2, 1, 1) else 16)) == 0, (l2, rad)
            else:
                assert (1 << l2) % ((1 << r) << log2T) == 0, (l2, rad)
            bits += r
        if planner == "cwt" and fused_ok(l2, 1, 1):
            assert rad[-1] == 7 and sum(rad[:-1]) >= 6, (l2, rad)  # the fused pass needs Ns >= 64 (fft_run)
        # the pruned generation reads spectrum (j0 >> S) + t (Q >> S): S <= log2 L - 7 whenever a 7-bit pass follows
        # the skipped ones
        for lvl in levels(l2)[1:] if planner == "cwt" else ():
            S = sum(rad[:lvl])
            assert S <= l2 - rad[lvl] and S >= 6, (l2, lvl)


def test_skip_thresholds_straddle_in_fp32():
    """The scales x (1 -+ 2^-12) around each threshold land on either side after rounding to fp32, and the straddling
    pair differs in its level by one."""
    for l2 in range(13, MAX_L2 + 1):
        for wav in ("gmw", "morlet"):
            for lvl in levels(l2)[1:]:
                t = threshold(l2, wav, lvl)
                lo, hi = f32(t * (1 - 2.0 ** -12)), f32(t * (1 + 2.0 ** -12))
                assert skip_level(l2, wav, float(lo)) == lvl - 1 and skip_level(l2, wav, float(hi)) == lvl, \
                    (l2, wav, lvl)
    # the issue's orders of magnitude: GMW level 1 from about 92, level 2 between 1 500 and 12 000; Morlet 3.2x
    assert 91 < threshold(20, "gmw", 1) < 93 and 94 < threshold(13, "gmw", 1) < 95 and 1600 < threshold(15, "gmw", 2) < 1700
    assert 11700 < threshold(27, "gmw", 2) < 11800
    assert abs(threshold(20, "morlet", 1) / threshold(20, "gmw", 1) - 14.5 / 4.5) < 1e-12


def test_case_table_reaches_every_cell():
    # cwt: every log2 L with both ends of its N range, every skip level of every plan for both wavelets
    seen = {}
    for l2, N, wavs in CWT_CASES:
        assert pad_len(N) == 1 << l2
        seen.setdefault(l2, set()).add(N)
        for wav in wavs:
            sc = case_scales(l2, N, wav)
            got = {skip_level(l2, wav, float(s)) for s in sc}
            assert got == set(levels(l2)), (l2, N, wav, got)
            # fused and stand-alone wherever the plan admits fused
            if fused_ok(l2, 1 << 20, 1):
                assert fused_ok(l2, N, len(sc)), (l2, N)
    assert sorted(seen) == list(range(2, 28)) and all(seen[l2] == set(n_range(l2)) for l2 in seen)
    for l2 in range(2, 28):
        wavs = {w for c in CWT_CASES if c[0] == l2 for w in c[2]}
        assert wavs == {"gmw", "morlet"}, l2
        # the unpad offset takes both parities
        assert {(pad_len(N) - N) // 2 % 2 for c in CWT_CASES if c[0] == l2 for N in [c[1]]} == {0, 1} or l2 <= 3, l2
    assert [fused_ok(l2, n_range(l2)[0], 6) for l2 in range(2, 28)] == [l2 in (14,) or l2 >= 18 for l2 in range(2, 28)]
    assert {fft_plan(l2)[0].__len__() for l2 in CWT_OPTION_CASES} == {1, 2, 3, 4}
    # rows path: every fft_plan_rows plan from 2^7 to 2^27, powers of two and Bluestein lengths
    # rows path: every plan its frames reach, 2^7 .. 2^17; the longest frames one tile takes, forward and inverse;
    # the plans of longer rows are fft_plan's, which the icwt cases below run
    assert (ROWS_SMEM, ROWS_FWD_MAX, ROWS_INV_MAX) == (200 * 1024, 45509, 51197)
    assert rows_tile_smem(ROWS_FWD_MAX // 2 + 1, 1, 1, True) <= ROWS_SMEM < rows_tile_smem(ROWS_FWD_MAX // 2 + 2, 1, 1, True)
    assert rows_tile_smem(ROWS_INV_MAX // 2 + 1, 1, 0, False) <= ROWS_SMEM < rows_tile_smem(ROWS_INV_MAX // 2 + 2, 1, 0, False)
    assert {rows_M(n) for n in ROWS_POW2} == {1 << k for k in range(11, 16)}
    assert [rows_M(n) for n in ROWS_BLUE] == [1 << k for k in range(7, 18)]
    assert all(n % 2 == 1 and rows_M(n) // 4 < n <= rows_M(n) // 2 and 32 < n <= ROWS_FWD_MAX for n in ROWS_BLUE)
    assert all(n > ROWS_FWD_MAX for n in ROWS_REFUSED) and any(n > ROWS_INV_MAX for n in ROWS_REFUSED)
    assert all(fft_plan_rows(l2) == fft_plan(l2) for l2 in range(13, 28))
    # icwt two-integral: every fft_plan M from 4 to 2^27, directly and through Bluestein
    Ms = [rows_M(n) if n & (n - 1) else n for n in ICWT2_LENS]
    assert set(Ms) == {1 << k for k in range(2, 28)}
    assert {rows_M(n) for n in ICWT2_LENS if n & (n - 1)} == {1 << k for k in range(3, 28)}
    # the fused -> stand-alone boundary
    l2b = pad_len(BOUNDARY_N).bit_length() - 1
    assert fused_ok(l2b, BOUNDARY_N, BOUNDARY_NS - 2) and not fused_ok(l2b, BOUNDARY_N, BOUNDARY_NS)
    assert (BOUNDARY_NS - 2) * BOUNDARY_N < 1 << 31 <= BOUNDARY_NS * BOUNDARY_N


def test_per_row_oracle_equals_the_whole_array_oracle():
    rng = np.random.default_rng(5)
    for N, wav, kw in ((1000, "gmw", {}), (3001, "morlet", dict(padtype="zero")), (700, "gmw", dict(rpadded=True)),
                       (513, "morlet", dict(l1_norm=False))):
        x = rng.standard_normal(N)
        sc = np.array([2.0, 9.3, N / 2.0])
        Wo, _, dWo = O.cwt(x, wav, sc, fs=4.0, derivative=True, **kw)
        rows = list(cwt_rows(x, wav, sc, dt=0.25, errors=True, **kw))
        for i, (W, dW, _) in enumerate(rows):
            assert np.abs(W - Wo[i]).max() <= 1e-12 * np.abs(Wo[i]).max(), (N, wav, kw)
            assert np.abs(dW - dWo[i]).max() <= 1e-12 * np.abs(dWo[i]).max(), (N, wav, kw)
        if not kw:
            eW, eD = P.cwt_row_errors(Wo, dWo, x, wav, sc, 0.25, "reflect")
            assert np.allclose([r[2][0] for r in rows], eW, rtol=1e-12, atol=0)
            assert np.allclose([r[2][1] for r in rows], eD, rtol=1e-12, atol=0)
    x = rng.standard_normal(5000)
    for n_fft, hop in ((1024, 300), (777, 5), (4096, 2048)):
        win = np.hanning(n_fft) + 0.1
        So, _ = O.stft(x, n_fft, hop, win, "reflect")
        assert np.abs(stft_frames(x, n_fft, hop, win) - So).max() <= 1e-12 * np.abs(So).max()
        assert np.abs(diff_window(win) - O.diff_window(win)).max() <= 1e-12 * np.abs(O.diff_window(win)).max()
        xo = O.istft(So, win, n_fft=n_fft, hop_len=hop, N=5000)
        assert np.abs(istft_ref(So, win, n_fft, hop, 5000) - xo).max() <= 1e-12 * np.abs(xo).max()
    for xl in (64, 777):
        Wx = rng.standard_normal((2, xl)) + 1j * rng.standard_normal((2, xl))
        sc = np.array([3.0, 7.0])
        for wav in ("gmw", "morlet"):
            xo = O.icwt(Wx, wav, sc, one_int=False)
            assert np.abs(icwt2_ref(Wx, wav, sc, xl) - xo).max() <= 1e-12 * np.abs(xo).max()


def test_per_row_check_catches_what_the_array_maximum_misses():
    """An oracle map of broadband input over scales 2 .. N/2: a 1e-3 error of the largest-scale row, relative to that
    row, passes rel() against the array maximum at the 1e-4 bar and fails the per-row check by far."""
    N = 1 << 14
    x = broadband(N, 3)
    sc = f32(2.0 ** np.linspace(1, np.log2(N / 2), 24))
    Wo, _, _ = O.cwt(x, "gmw", sc)
    bad = Wo.copy()
    rng = np.random.default_rng(0)
    bad[-1] += 1e-3 * np.abs(Wo[-1]).max() * np.exp(2j * np.pi * rng.random(N))
    assert np.abs(bad - Wo).max() / np.abs(Wo).max() < 1e-4  # the array-maximum check stays green
    l2, mx = row_ratios(bad[-1], Wo[-1])
    assert l2 > 10 * B_L2 and mx > 5 * B_MAX
    assert all(row_ratios(bad[i], Wo[i]) == (0.0, 0.0) for i in range(len(sc) - 1))


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _engine():
    from ssqueeze_rs_b200.batch import Engine
    return Engine(0)


def _free(*objs):
    import torch
    gc.collect()
    torch.cuda.empty_cache()


def _col_slices(N, l2):
    if l2 < SLICE_FROM_L2:
        return [slice(0, N)]
    w = 1 << 16
    return [slice(0, w), slice(N // 2 - w // 2, N // 2 + w // 2), slice(N - w, N)]


def _classify_slices(tag, wav, sc, sf, N, rows_ref, kb, w_dev, Tx, slices, check_tx=True):
    """Bins of the device (kb, w of one channel, numpy) against the oracle rows on each column slice; Tx per Tx row
    against the oracle's W accumulated over the device's bins (`reaccumulate_cwt`)."""
    ns = len(sc)
    eW = np.array([r[2][0] for r in rows_ref])
    eD = np.array([r[2][1] for r in rows_ref])
    for s in slices:
        Ws = np.stack([r[0][s] for r in rows_ref])
        dWs = np.stack([r[1][s] for r in rows_ref])
        w_o = O.phase_cwt(Ws, dWs, GAMMA)
        _, k_o = O.ssqueeze_cwt(Ws, w_o, sf, "sum", True)
        ao = dict(Wx=Ws, dWx=dWs, w=w_o, k=k_o, scales=sc)
        rep = P.classify_cwt_bins(kb[:, s], ao, None, wav, 1.0, "reflect", sf, w_dev=w_dev[:, s], row_err=(eW, eD))
        pub = P.public(rep)
        assert rep["unexplained"] == 0, (tag, s, pub)
        assert rep["max_err_over_tol"] <= 1.0, (tag, s, pub)
        if check_tx:
            # each contribution of scale row i to a Tx element is held to max |W_i|: the bound of element (k, j) is
            # B_MAX times the sum of max |W_i| over the rows the device added there
            kbs = kb[:, s].astype(np.int64)
            Tref = P.reaccumulate_cwt(Ws, kbs, ns)
            A = np.abs(P.reaccumulate_cwt(np.repeat(np.abs(Ws).max(axis=1, keepdims=True), Ws.shape[1], axis=1)
                                          + 0j, kbs, ns))
            e = np.abs(Tx[:, s].astype(np.complex128) - Tref)
            assert not e[A == 0].any(), tag
            r = float((e[A > 0] / A[A > 0]).max()) if (A > 0).any() else 0.0
            w = WORST.setdefault("ssq_cwt Tx", [0.0, 0.0, ""])
            w[1] = max(w[1], r)
            assert r <= BOUNDS["ssq_cwt Tx"][1], (tag, r)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: cwt and ssq_cwt on every plan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("l2,N,wavs", CWT_CASES, ids=_ids(CWT_CASES))
def test_cwt_and_ssq_cwt_on_every_plan(l2, N, wavs):
    """W and dW of every row against the per-row oracle; ssq_cwt fused (where cwt_fused_ok holds) and stand-alone,
    same bins bit for bit, every bin classified, Tx per Tx row."""
    import torch
    eng = _engine()
    x = broadband(N, 1000 + l2 * 2 + (N & 1))
    xd = torch.from_numpy(x.astype(np.float32)).cuda().view(1, -1)
    slices = _col_slices(N, l2)
    for wav in wavs:
        sc = case_scales(l2, N, wav)
        ns = len(sc)
        W, dW = eng.cwt(xd, wav, sc, derivative=True)
        torch.cuda.synchronize()
        assert eng.last_kernel_name() == "fft_pass_kernel"
        runs = {}
        for fused in ((True, False) if fused_ok(l2, N, ns) else (False,)):
            eng.ctx.set_option("no_cwt_fused", 0 if fused else 1)
            try:
                Tx, sf, aux = eng.ssq_cwt(xd, wav, sc, maprange="maximal", return_aux=True, return_freqs=True)
                torch.cuda.synchronize()
                name = eng.last_kernel_name()
            finally:
                eng.ctx.set_option("no_cwt_fused", 0)
            assert ("fused" in name) if fused else ("reassign" in name), (fused, name)
            runs[fused] = (Tx[0], aux["kb"][0], aux["w"][0])
            del aux
        if len(runs) == 2:
            assert torch.equal(runs[True][1], runs[False][1])  # same W, dW bits -> same bins
        sfo = O.ssq_freqs_cwt(ns, 1.0 / N, 0.5, "log")
        assert np.allclose(sf, sfo, rtol=1e-13)
        rows_ref = []
        for i, (Wr, dWr, err) in enumerate(cwt_rows(x, wav, sc, errors=True)):
            what = f"L=2^{l2} N={N} {wav} scale={sc[i]:.9g} level={skip_level(l2, wav, float(sc[i]))}"
            check_row("cwt W", W[0, i].cpu().numpy(), Wr, what, floor=err[2])
            check_row("cwt dW", dW[0, i].cpu().numpy(), dWr, what, floor=err[3])
            rows_ref.append((Wr, dWr, err) if len(slices) == 1 else
                            (np.concatenate([Wr[s] for s in slices]), np.concatenate([dWr[s] for s in slices]), err))
            del Wr, dWr
        del W, dW
        _free()
        # slices index the concatenated slice columns from here on
        if len(slices) > 1:
            w = slices[0].stop - slices[0].start
            cat = [slice(j * w, (j + 1) * w) for j in range(len(slices))]
        else:
            cat = slices
        for fused, (Tx, kb, wd) in runs.items():
            def cols(t):
                return torch.cat([t[:, s] for s in slices], dim=1).cpu().numpy() if len(slices) > 1 else t.cpu().numpy()
            _classify_slices((l2, N, wav, fused), wav, sc, sfo, N, rows_ref, cols(kb), cols(wd), cols(Tx), cat)
        del runs, rows_ref
        _free()


@pytest.mark.gpu
@pytest.mark.parametrize("l2", CWT_OPTION_CASES)
def test_cwt_options_per_pass_count(l2):
    """l1_norm=False, padtype="zero" and rpadded=True on one size per pass count (1 .. 4 passes), per row."""
    import torch
    eng = _engine()
    N = n_range(l2)[0]
    x = broadband(N, 77 + l2)
    xd = torch.from_numpy(x.astype(np.float32)).cuda().view(1, -1)
    sc = case_scales(l2, N, "gmw")
    for kw in (dict(l1_norm=False), dict(padtype="zero"), dict(rpadded=True)):
        W, dW = eng.cwt(xd, "gmw", sc, derivative=True, **kw)
        torch.cuda.synchronize()
        assert eng.last_kernel_name() == "fft_pass_kernel"
        for i, (Wr, dWr, err) in enumerate(cwt_rows(x, "gmw", sc, errors=True, **kw)):
            what = f"L=2^{l2} {kw} scale={sc[i]:.9g}"
            f = 1.0 if kw.get("l1_norm", True) else math.sqrt(sc[i])
            check_row("cwt W", W[0, i].cpu().numpy(), Wr, what, floor=err[2] * f)
            check_row("cwt dW", dW[0, i].cpu().numpy(), dWr, what, floor=err[3] * f)
        del W, dW
        _free()


@pytest.mark.gpu
def test_cwt_row_blocks_at_2_27():
    """3 channels of 89 478 485 samples (L = 2^27): cwt_forward and cwt_inverse_rows launch at most 2 rows at this
    length, so the batch crosses row blocks; every channel equals its one-channel call (W, dW bit for bit; the fused
    tail: equal bins, Tx within 1e-5 of each row's maximum)."""
    import torch
    from test_at_scale import _signals
    eng = _engine()
    N = n_range(27)[1]
    x = _signals(3, N, 27)
    sc = f32([2.0, threshold(27, "gmw", 2) * (1 + 2.0 ** -12)])
    W, dW = eng.cwt(x, "gmw", sc, derivative=True)
    torch.cuda.synchronize()
    for c in range(3):
        Wc, dWc = eng.cwt(x[c:c + 1], "gmw", sc, derivative=True)
        assert torch.equal(Wc[0], W[c]) and torch.equal(dWc[0], dW[c]), c
        del Wc, dWc
    del W, dW
    _free()
    Tx, _, aux = eng.ssq_cwt(x, "gmw", sc, return_aux=True)
    torch.cuda.synchronize()
    assert "fused" in eng.last_kernel_name(), eng.last_kernel_name()
    kb = aux["kb"]
    del aux
    for c in range(3):
        Tc, _, ac = eng.ssq_cwt(x[c:c + 1], "gmw", sc, return_aux=True)
        assert torch.equal(ac["kb"][0], kb[c]), c
        lim = 1e-5 * Tc[0].abs().amax(dim=1, keepdim=True)
        assert bool(((Tx[c] - Tc[0]).abs() <= lim).all()), c
        del Tc, ac
    del Tx, kb, x
    _free()


@pytest.mark.gpu
def test_ssq_cwt_fused_to_standalone_boundary():
    """ns N >= 2^31 sends ssq_cwt to the stand-alone path: N = 2^22 with 513 scales (stand-alone) and the first 511
    of them (fused); sampled rows classified against the oracle on column slices in both, and their phase transform
    agrees between the two paths."""
    import torch
    N, ns = BOUNDARY_N, BOUNDARY_NS
    l2 = pad_len(N).bit_length() - 1
    eng = _engine()
    x = broadband(N, 2222)
    xd = torch.from_numpy(x.astype(np.float32)).cuda().view(1, -1)
    sc = f32(2.0 ** np.linspace(1, np.log2(N / 2), ns))
    rows = [0, 1, 255, 509, 510]
    slices = [slice(0, 1 << 14), slice(N // 2, N // 2 + (1 << 14)), slice(N - (1 << 14), N)]
    ref = {i: r for i, r in zip(rows, cwt_rows(x, "gmw", sc[rows], errors=True))}
    got = {}
    for n_sc, expect in ((ns, "reassign"), (ns - 2, "fused")):
        assert fused_ok(l2, N, n_sc) == (expect == "fused")
        Tx, sf, aux = eng.ssq_cwt(xd, "gmw", sc[:n_sc], maprange="maximal", return_aux=True, return_freqs=True)
        torch.cuda.synchronize()
        assert expect in eng.last_kernel_name(), eng.last_kernel_name()
        del Tx
        ri = torch.as_tensor(rows, device="cuda")
        kb = aux["kb"][0][ri].cpu().numpy()
        wd = aux["w"][0][ri].cpu().numpy()
        del aux
        _free()
        sfo = O.ssq_freqs_cwt(n_sc, 1.0 / N, 0.5, "log")
        assert np.allclose(sf, sfo, rtol=1e-13)
        rows_ref = [ref[i] for i in rows]
        _classify_slices(("boundary", n_sc), "gmw", sc[rows], sfo, N, rows_ref, kb, wd, None, slices, check_tx=False)
        got[n_sc] = wd
    a, b = got[ns], got[ns - 2]
    fin = np.isfinite(a) & np.isfinite(b)
    assert np.array_equal(np.isfinite(a), np.isfinite(b))
    assert np.all(np.abs(a[fin] - b[fin]) <= 4 * EPS32 * np.abs(b[fin]))
    del xd
    _free()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the STFT rows path and the two-integral icwt on every plan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", ROWS_POW2 + ROWS_BLUE)
def test_rows_path_every_plan(n_fft):
    """3 frames (hop n_fft / 2) of 2 channels through Engine.stft, per frame against rfft of the windowed frame;
    ssq_stft: Sx, dSx per frame and every bin classified up to n_fft 2^14 (the oracle's arg-min over the whole grid is
    quadratic in n_fft), w where |Sx| carries the frame above; istft of the device's Sx against the oracle.
    Bluestein: the library builds its filter with a double-precision DFT on the host."""
    import torch
    from ssqueeze_rs_b200 import _lib, _rs
    pow2 = n_fft & (n_fft - 1) == 0
    kernel = "fft_pass rows" if pow2 else "bluestein fft_pass rows"
    fam = "rows" if pow2 else "bluestein"
    eng = _engine()
    n, hop = n_fft + 1, n_fft // 2
    xs = [broadband(n, 5000 + n_fft + c) for c in range(2)]
    xd = torch.from_numpy(np.stack(xs).astype(np.float32)).cuda()
    win = f32(np.hanning(n_fft) + 0.05)
    Sx = eng.stft(xd, win, n_fft, hop)
    torch.cuda.synchronize()
    assert eng.last_kernel_name().startswith(kernel + " + stft_generic_kernel<rows>"), eng.last_kernel_name()
    for c in range(2):
        So = stft_frames(xs[c], n_fft, hop, win)
        Sc = Sx[c].cpu().numpy()
        assert Sc.shape == So.shape
        for f in range(So.shape[1]):
            check_row(f"stft {fam}", Sc[:, f], So[:, f], f"n_fft={n_fft} ch={c} frame={f}")
        # istft of the device's Sx
        xr = eng.istft(Sx[c:c + 1], win, n_fft, hop, N=n)
        torch.cuda.synchronize()
        assert eng.last_kernel_name().startswith(kernel + " + istft_ola_kernel<rows>"), eng.last_kernel_name()
        check_row(f"istft {fam}", xr[0].cpu().numpy(), istft_ref(Sc.astype(np.complex128), win, n_fft, hop, n),
                  f"n_fft={n_fft} ch={c}")
        del So, Sc, xr
    del Sx, xd
    _free()
    # ssq_stft (float64 entry point, diagnostic variant of the same kernels)
    x = xs[0]
    if n_fft <= CLASSIFY_STFT_MAX:
        from test_parity_stft import check_ssq
        rep = check_ssq(x, win, n_fft, hop, 1.0, expect_kernel=kernel)
        assert rep["unexplained"] == 0
    Tx, sf, aux = _rs.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=1.0, return_aux=True)
    assert _lib.default_context().last_kernel_name().startswith(kernel), _lib.default_context().last_kernel_name()
    del Tx
    So = stft_frames(x, n_fft, hop, win)
    dSo = stft_frames(x, n_fft, hop, diff_window(win))
    for f in range(So.shape[1]):
        check_row(f"ssq_stft Sx {fam}", aux["Sx"][:, f], So[:, f], f"n_fft={n_fft} frame={f}")
        check_row(f"ssq_stft dSx {fam}", aux["dSx"][:, f], dSo[:, f], f"n_fft={n_fft} frame={f}")
    if n_fft > CLASSIFY_STFT_MAX:
        # w where |Sx| is at least 10 % of the frame's maximum: within 1e-2 of a bin of the oracle's
        w_o = O.phase_stft(So, dSo, np.linspace(0.0, 0.5, n_fft // 2 + 1), GAMMA)
        big = np.abs(So) >= 0.1 * np.abs(So).max(axis=0, keepdims=True)
        assert big.any()
        err = np.abs(aux["w"][big] - w_o[big]) * n_fft
        assert float(err.max()) <= 1e-2, float(err.max())
    del aux, So, dSo


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", ROWS_REFUSED)
def test_rows_path_refuses_frames_past_one_tile(n_fft):
    """Frames longer than one tile of shared memory takes: stft, ssq_stft and istft are SSQ_EUNSUPPORTED with the
    limit in the message, before anything is launched."""
    import torch
    from ssqueeze_rs_b200 import _rs
    from ssqueeze_rs_b200._lib import SsqError
    eng = _engine()
    x = broadband(64, n_fft)
    win = np.ones(n_fft)
    with pytest.raises(SsqError, match=f"n_fft={n_fft}: .* n_fft <= {ROWS_FWD_MAX}"):
        eng.stft(torch.from_numpy(x.astype(np.float32)).cuda().view(1, -1), win, n_fft, n_fft // 2)
    with pytest.raises(SsqError, match=f"n_fft <= {ROWS_FWD_MAX}"):
        _rs.ssq_stft(x, win, n_fft=n_fft, hop_len=n_fft // 2)
    if n_fft // 2 + 1 > ROWS_INV_MAX // 2 + 1:
        Sx = torch.zeros((1, n_fft // 2 + 1, 2), dtype=torch.complex64, device="cuda")
        with pytest.raises(SsqError, match=f"n_fft={n_fft}: .* n_fft <= {ROWS_INV_MAX}"):
            eng.istft(Sx, win, n_fft, n_fft // 2, N=64)
        del Sx
    _free()


@pytest.mark.gpu
@pytest.mark.parametrize("x_len", ICWT2_LENS)
def test_icwt_two_integral_every_plan(x_len):
    """icwt(one_int=False) of a random fp32 map of 2 scales whose bands fall on bins of the row, against the
    oracle relative to the output's norm."""
    from ssqueeze_rs_b200 import _lib, _rs
    pow2 = x_len & (x_len - 1) == 0
    rng = np.random.default_rng(x_len)
    wav = "morlet" if rows_M(x_len).bit_length() % 2 else "gmw"
    centre = 2.7144176165949063 if wav == "gmw" else 6.0
    k1, k2 = max(1, x_len // 5), max(1, x_len // 17)
    sc = f32([centre * x_len / (2 * math.pi * k1), centre * x_len / (2 * math.pi * k2) * (1.1 if k1 == k2 else 1.0)])
    Wx = (rng.standard_normal((2, x_len)) + 1j * rng.standard_normal((2, x_len))).astype(np.complex64)
    Wx = Wx.astype(np.complex128)
    xr = _rs.icwt(Wx, wav, sc, one_int=False)
    name = _lib.default_context().last_kernel_name()
    assert name == ("icwt2_accum_kernel" if pow2 else "icwt2_accum_kernel<bluestein>"), name
    check_row("icwt2" if pow2 else "icwt2 bluestein", xr, icwt2_ref(Wx, wav, sc, x_len), f"x_len={x_len} {wav}")
    del Wx, xr

"""GPU parity: the CUDA path (through the C ABI, via the `_rs` mirror) against
the float64 oracle on the same seeded inputs.

Tolerances (north star): |Sx|, |Tx| and reconstructions within rtol 1e-4 of the
array maximum in fp32; reassignment bin indices identical except where w falls
within fp32 rounding of a bin edge -- such cases are counted and bounded.
"""
import os

import numpy as np
import pytest

from oracle import parity as P
from oracle import ssq_oracle as O

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
RTOL = 1e-4


def _rs():
    from ssqueeze_rs_b200 import _rs
    return _rs


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def check_ssq(x, win, n_fft, hop, fs, padtype="reflect", squeezing="sum", gamma=None, modulated=False,
              expect_kernel=None, oracle_out=None):
    """Full parity report of one ssq_stft call.  The destination bin of every (source bin, frame) comes from the
    SAME kernel that produced Tx (the diagnostic compile-time variant: `kb`, plus Sx, dSx, w); every bin that
    differs from the oracle's arg-min (ssq_stft.rs:276-301) must be explained by the fp32 bin-edge gate of
    oracle/parity.py, and Tx must be the reference's accumulation over exactly those bins."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    kw = dict(n_fft=n_fft, hop_len=hop, fs=fs, padtype=padtype, squeezing=squeezing, gamma=gamma, modulated=modulated)
    Tx, sf, aux = rs.ssq_stft(x, win, return_aux=True, **kw)
    name = _lib.default_context().last_kernel_name()
    if expect_kernel:
        assert expect_kernel in name, name
    Tx_plain, _ = rs.ssq_stft(x, win, **kw)
    assert _lib.default_context().last_kernel_name() == name
    assert np.array_equal(Tx, Tx_plain), "diagnostic variant and production kernel disagree: " + name
    Tx_o, sf_o, ao = oracle_out if oracle_out is not None else O.ssq_stft(x, win, return_aux=True, **kw)
    assert Tx.shape == Tx_o.shape and Tx.dtype == np.complex128 and sf.dtype == np.float64
    assert np.allclose(sf, sf_o, rtol=1e-15, atol=0)
    assert rel(aux["Sx"], ao["Sx"]) < RTOL, ("Sx", rel(aux["Sx"], ao["Sx"]))
    assert rel(aux["dSx"], ao["dSx"]) < 2 * RTOL, ("dSx", rel(aux["dSx"], ao["dSx"]))
    kb = aux["kb"]
    rep = P.classify_stft_bins(kb, ao, n_fft, fs, gamma, w_dev=aux["w"])
    pub = P.public(rep)
    pub["kernel"] = name
    assert rep["unexplained"] == 0, pub
    assert rep["max_err_over_tol"] <= 1.0, pub  # the device's w sits inside the derived fp32 bound everywhere
    # Tx = the reference's accumulation of Sx over exactly the bins the kernel reports
    Tref = P.reaccumulate(ao["Sx"], kb, fs, squeezing)
    assert rel(Tx, Tref) < RTOL, ("Tx vs oracle Sx accumulated over the device's bins", rel(Tx, Tref), pub)
    # columns without any flip agree with the oracle's Tx element by element
    good_cols = ~(kb != ao["k"]).any(axis=0)
    if good_cols.any():
        assert rel(Tx[:, good_cols], Tx_o[:, good_cols]) < RTOL, pub
    pub["good_cols"] = int(good_cols.sum())
    return pub


def test_readme_sine_config1():
    """BASELINE config 1: 1 s 100 Hz sine, fs=1 kHz, n_fft=256 hop=64 Hann."""
    rs = _rs()
    z = np.load(os.path.join(G, "readme_cases.npz"))
    x = z["x"]
    win = np.hanning(256)
    Sx, freqs = rs.stft(x, 256, 64, win, "reflect")
    assert Sx.shape == (129, 16) and freqs.shape == (129,) and Sx.dtype == np.complex128
    assert np.allclose(freqs, z["stft_freqs"])
    assert rel(Sx, z["stft_Sx"]) < RTOL
    xr = rs.istft(Sx, win, n_fft=256, hop_len=64, N=len(x))
    assert np.abs(xr - x).max() < 2e-5
    assert np.abs(xr - z["istft_x"]).max() < 2e-5
    Tx, sf = rs.ssq_stft(x, window=win, n_fft=256, hop_len=64, fs=1000, padtype="reflect", squeezing="sum")
    assert Tx.shape == (129, 16) and sf.shape == (129,)
    # a pure tone is the worst fp32 case for w (SURVEY 7): compare energy per column
    To = z["ssq_stft_Tx"]
    assert np.abs(np.abs(Tx).sum(0) - np.abs(To).sum(0)).max() < 1e-3 * np.abs(To).sum(0).max()
    k_g, k_o = np.abs(Tx).argmax(0), np.abs(To).argmax(0)
    assert np.array_equal(k_g, k_o)
    assert rel(Tx[k_o, np.arange(16)], To[k_o, np.arange(16)]) < 1e-3


@pytest.mark.parametrize("n_fft,hop,N", [(256, 64, 1000), (512, 32, 6000), (64, 8, 777), (128, 1, 300),
                                         (1024, 100, 5000), (32, 7, 100), (2048, 512, 9000)])
def test_ssq_stft_noise_pow2(n_fft, hop, N):
    rng = np.random.default_rng(n_fft + hop)
    x = rng.standard_normal(N)
    rep = check_ssq(x, np.hanning(n_fft), n_fft, hop, fs=30000.0)
    assert rep["mismatch_above_energy_gate"] <= max(2, rep["bins_total"] // 2000), rep


@pytest.mark.parametrize("n_fft,hop,N", [(255, 7, 1000), (129, 1, 300), (65, 3, 400), (120, 2, 129), (121, 3, 128)])
def test_ssq_stft_non_pow2(n_fft, hop, N):
    rng = np.random.default_rng(n_fft)
    x = rng.standard_normal(N)
    win = np.hanning(n_fft + 2)[1:-1].copy()
    check_ssq(x, win, n_fft, hop, fs=1.0)


@pytest.mark.parametrize("n_fft,hop,N", [(500, 125, 6000), (1000, 100, 5000), (3000, 750, 20000), (8192, 2048, 40000),
                                         (6000, 1500, 30000), (16384, 8192, 50000), (4097, 1000, 9000)])
def test_ssq_stft_any_length_rows_path(n_fft, hop, N):
    """The reference takes any n_fft (rustfft, ssq_stft.rs:92,198-199): lengths above 4096 and lengths that are not
    powers of two run through the batched row FFT (Bluestein for the latter), then the same split / phase transform /
    reassignment; every bin classified against the oracle, stft and the istft of the result as well."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(n_fft)
    x = rng.standard_normal(N) * 3.0
    win = np.hanning(n_fft + 2)[1:-1].copy()
    rep = check_ssq(x, win, n_fft, hop, fs=1000.0, expect_kernel="rows")
    assert rep["unexplained"] == 0
    check_ssq(x, win, n_fft, hop, fs=1000.0, expect_kernel="rows", padtype="zero", squeezing="lebesgue")
    check_ssq(x, win, n_fft, hop, fs=1000.0, expect_kernel="rows", modulated=True)
    Sx, _ = rs.stft(x, n_fft, hop, win, "reflect")
    assert "rows" in _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, n_fft, hop, win, "reflect")
    assert rel(Sx, So) < RTOL, rel(Sx, So)
    # the inverse through the same row passes: against the oracle on a modified spectrum, and the round trip
    Sm = So * (1 + 0.05 * rng.standard_normal(So.shape))
    for wexp in (1, 0):
        xr = rs.istft(Sm, win, n_fft=n_fft, hop_len=hop, N=N, win_exp=wexp)
        assert "rows" in _lib.default_context().last_kernel_name()
        xo = O.istft(Sm, win, n_fft=n_fft, hop_len=hop, N=N, win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30), (n_fft, wexp)
    if hop * 2 <= n_fft:
        xb = rs.istft(Sx, win, n_fft=n_fft, hop_len=hop, N=N)
        assert np.abs(xb - x).max() < 1e-4 * np.abs(x).max()


def test_ssq_stft_vs_upstream_golden():
    z = np.load(os.path.join(G, "upstream_odd.npz"))
    rs = _rs()
    for ci, (N, n_fft, hop) in enumerate(z["cases"]):
        p = f"c{ci}_"
        Tx, sf, aux = rs.ssq_stft(z[p + "x"], z[p + "window"], n_fft=int(n_fft), hop_len=int(hop), fs=1.0,
                                  return_aux=True)
        assert rel(aux["Sx"], z[p + "Sx"]) < RTOL
        assert rel(aux["dSx"], z[p + "dSx"]) < 2 * RTOL
        To = z[p + "Tx"]
        bad = np.abs(Tx - To) > RTOL * np.abs(To).max()
        assert bad.mean() < 2e-3, bad.mean()
        assert np.abs(Tx.sum(0) - To.sum(0)).max() < 1e-3 * np.abs(To).max()


def test_benchmark_geometry_vs_upstream_golden():
    """n_fft=512, hop=32 (the benchmarked kernel) directly against upstream's output on the frames that touch
    no padding (tests/golden/upstream_even512.npz; see make_golden.py for the one-sample shift)."""
    z = np.load(os.path.join(G, "upstream_even512.npz"))
    rs = _rs()
    j0, j1 = z["cols"]
    Tx, sf, aux = rs.ssq_stft(z["x"], z["window"], n_fft=512, hop_len=32, fs=1.0, return_aux=True)
    assert rel(aux["Sx"][:, j0:j1], z["Sx"]) < RTOL
    assert rel(aux["dSx"][:, j0:j1], z["dSx"]) < 2 * RTOL
    To = z["Tx"]
    bad = np.abs(Tx[:, j0:j1] - To) > RTOL * np.abs(To).max()
    assert bad.mean() < 2e-3, bad.mean()
    assert np.abs(Tx[:, j0:j1].sum(0) - To.sum(0)).max() < 1e-3 * np.abs(To).max()
    assert np.allclose(sf, z["ssq_freqs"], rtol=0, atol=1e-15)


def test_ssq_stft_options():
    rng = np.random.default_rng(5)
    x = rng.standard_normal(2000)
    win = np.hanning(128)
    check_ssq(x, win, 128, 16, fs=1.0, padtype="zero")
    check_ssq(x, win, 128, 16, fs=250.0, squeezing="lebesgue")
    check_ssq(x, win, 128, 16, fs=250.0, gamma=5.0)       # a gate that actually bites
    check_ssq(x, win, 128, 16, fs=250.0, padtype="bogus")  # silent fallback to reflect
    check_ssq(x, win, 128, 1, fs=1.0, modulated=True)
    check_ssq(x, np.hanning(100), 128, 16, fs=1.0)          # window centre-padded to n_fft
    check_ssq(x, np.hanning(64), 256, 300, fs=1.0)          # hop > n_fft
    check_ssq(x, win, 128, 16, fs=250.0, gamma=-1.0)        # explicit negative gamma: nothing is gated (ssq_stft.rs:23)
    check_ssq(x * 1e-17, win, 128, 16, fs=250.0, gamma=-1.0)  # ... even where the default gamma would gate everything


def test_short_and_ragged_inputs():
    rs = _rs()
    rng = np.random.default_rng(6)
    for N, n_fft, hop in [(1, 16, 1), (2, 16, 3), (5, 64, 2), (31, 32, 32), (33, 32, 32), (100, 512, 32)]:
        x = rng.standard_normal(N)
        win = np.hanning(n_fft)
        Sx, _ = rs.stft(x, n_fft, hop, win, "reflect")
        So, _ = O.stft(x, n_fft, hop, win, "reflect")
        assert Sx.shape == So.shape
        assert rel(Sx, So) < RTOL
        Tx, sf = rs.ssq_stft(x, win, n_fft=n_fft, hop_len=hop)
        To, sfo = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop)
        assert Tx.shape == To.shape
        assert np.abs(Tx.sum(0) - To.sum(0)).max() < 1e-3 * max(np.abs(To).max(), 1e-30)


def test_stft_window_semantics_and_errors():
    rs = _rs()
    from ssqueeze_rs_b200 import PanicException
    x = np.random.default_rng(7).standard_normal(500)
    # stft does NOT fit the window: longer window -> first n_fft taps (stft_utils.rs:8)
    win = np.hanning(80)
    Sx, _ = rs.stft(x, 64, 16, win, "zero")
    So, _ = O.stft(x, 64, 16, win, "zero")
    assert rel(Sx, So) < RTOL
    with pytest.raises(PanicException):
        rs.stft(x, 64, 16, np.hanning(32), "reflect")  # rustfft length panic
    with pytest.raises(PanicException):
        rs.stft(x, 64, 0, np.hanning(64), "reflect")   # division by zero (stft.rs:33)
    with pytest.raises(PanicException):
        rs.ssq_stft(np.zeros(0), np.hanning(8), n_fft=8)
    with pytest.raises(ValueError):
        rs.ssq_stft(x, np.hanning(128), n_fft=64)
    # n_fft default = min(len(x), 512) (ssq_stft.rs:92)
    Tx, sf = rs.ssq_stft(x, np.hanning(100))
    assert Tx.shape == (500 // 2 + 1, 500)


@pytest.mark.parametrize("N", [128, 129])
@pytest.mark.parametrize("n_fft", [120, 121, 128])
@pytest.mark.parametrize("hop", [1, 2, 3])
def test_stft_istft_roundtrip(N, n_fft, hop):
    """old/tests/reconstruction_test.py:160-179 re-hosted (fp32 threshold)."""
    rs = _rs()
    x = np.random.default_rng(N * n_fft + hop).standard_normal(N)
    win = np.hanning(n_fft + 2)[1:-1].copy()
    Sx, _ = rs.stft(x, n_fft, hop, win, "reflect")
    xr = rs.istft(Sx, win, n_fft=n_fft, hop_len=hop, N=N)
    assert len(xr) == N
    assert np.abs(x - xr).mean() < 5e-6
    xo = O.istft(Sx, win, n_fft=n_fft, hop_len=hop, N=N)
    assert np.abs(xr - xo).max() < RTOL * max(1.0, np.abs(xo).max())


def test_istft_options_vs_oracle():
    rs = _rs()
    rng = np.random.default_rng(11)
    x = rng.standard_normal(3000)
    for n_fft, hop, wexp in [(512, 32, 1), (512, 32, 0), (256, 64, 2), (64, 64, 1), (100, 25, 1)]:
        win = np.hanning(n_fft + 2)[1:-1].copy()
        So, _ = O.stft(x, n_fft, hop, win, "reflect")
        So = So * (1 + 0.1 * rng.standard_normal(So.shape))  # a *modified* STFT (Griffin-Lim case)
        xr = rs.istft(So, win, n_fft=n_fft, hop_len=hop, N=len(x), win_exp=wexp)
        xo = O.istft(So, win, n_fft=n_fft, hop_len=hop, N=len(x), win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * np.abs(xo).max(), (n_fft, hop, wexp)
    # N omitted: hop * n_frames samples (_stft.py:231)
    So, _ = O.stft(x, 128, 16, np.hanning(128), "reflect")
    assert len(rs.istft(So, np.hanning(128), hop_len=16)) == 16 * So.shape[1]


def test_issq_stft_roundtrip():
    """old/tests/reconstruction_test.py:182-206 re-hosted: MAE < 0.1."""
    rs = _rs()
    for N in (128, 129):
        x = np.random.default_rng(N).standard_normal(N)
        for n_fft in (120, 128):
            win = np.hanning(n_fft + 2)[1:-1].copy()
            for fs in (1.0, 250.0):
                Tx, _ = rs.ssq_stft(x, win, n_fft=n_fft, hop_len=1, fs=fs, modulated=True)
                y = rs.issq_stft(Tx, win, n_fft=n_fft, hop_len=1, fs=fs)
                yo = O.issq_stft(O.ssq_stft(x, win, n_fft=n_fft, hop_len=1, fs=fs, modulated=True)[0], win,
                                 n_fft=n_fft, hop_len=1, fs=fs)
                assert np.abs(y - yo).max() < 1e-3 * np.abs(yo).max()
                sh = n_fft // 2 - (n_fft - 1) // 2  # y[j] ~ x[j + sh]
                mae = np.abs(y[:N - sh] - x[sh:]).mean()
                assert mae < 0.1, (N, n_fft, mae)
    with pytest.raises(ValueError):
        rs.issq_stft(np.zeros((65, 10), dtype=np.complex128), np.hanning(128), hop_len=2)


# ---------------------------------------------------------------------------
# fast path (n_fft=512 register-resident kernel) and the batched device API
# ---------------------------------------------------------------------------

def _flip_tolerant_compare(Tx, To, max_bad_frac=2e-3):
    """Cross-KERNEL agreement only (two CUDA kernels on the same input: different rounding -> a few edge flips).
    Parity against the oracle goes through check_ssq / check_ssq_device, which classify every flip."""
    sc = np.abs(To).max()
    assert np.abs(Tx.sum(0) - To.sum(0)).max() < 20 * RTOL * sc
    bad = np.abs(Tx - To) > RTOL * sc
    assert bad.mean() < max_bad_frac, bad.mean()
    cols_ok = ~bad.any(axis=0)
    assert cols_ok.mean() > 0.5
    assert rel(Tx[:, cols_ok], To[:, cols_ok]) < RTOL
    return float(bad.mean())


def check_ssq_device(eng, xd, win, n_fft, hop, fs, channels=None, frame_slices=None, expect_kernel=None,
                     framing="crate", **kw):
    """check_ssq for the batched device API (Engine): the diagnostic twin runs on the whole batch; the oracle runs per
    channel, or -- for recordings too long for it -- on slices of frames (a frame depends on its own n_fft samples
    only, so the oracle is run on the samples of the slice and its interior frames are compared).
    frame_slices: list of (channel, first_frame, n_frames_in_slice).  framing: the oracle's framing ("upstream" for
    an engine whose context has upstream_framing set)."""
    import torch
    Tx, aux = eng.ssq_stft(xd, win, n_fft, hop, fs, return_aux=True, **kw)
    name = eng.last_kernel_name()
    if expect_kernel:
        assert expect_kernel in name, name
    Tx_plain = eng.ssq_stft(xd, win, n_fft, hop, fs, **kw)
    torch.cuda.synchronize()
    assert torch.equal(Tx, Tx_plain), "diagnostic variant and production kernel disagree: " + name
    okw = dict(n_fft=n_fft, hop_len=hop, fs=fs, return_aux=True, framing=framing, **kw)
    total = dict(bins_total=0, mismatch_total=0, within_edge=0, ill_conditioned=0, below_energy_gate=0, gate_edge=0,
                 unexplained=0, max_err_over_tol=0.0)

    def one(kb, w, T, To, ao):
        rep = P.classify_stft_bins(kb, ao, n_fft, fs, kw.get("gamma"), w_dev=w)
        assert rep["unexplained"] == 0, P.public(rep)
        assert rep["max_err_over_tol"] <= 1.0, P.public(rep)
        Tref = P.reaccumulate(ao["Sx"], kb, fs, kw.get("squeezing", "sum"))
        assert rel(T, Tref) < RTOL, ("Tx vs oracle Sx over the device's bins", rel(T, Tref))
        good = ~(kb != ao["k"]).any(axis=0)
        if good.any():
            assert rel(T[:, good], To[:, good]) < RTOL
        for k in total:
            total[k] = max(total[k], rep[k]) if k == "max_err_over_tol" else total[k] + rep[k]

    if frame_slices is None:
        for c in (range(xd.shape[0]) if channels is None else channels):
            To, _, ao = O.ssq_stft(xd[c].cpu().numpy().astype(np.float64), win, **okw)
            one(aux["kb"][c].cpu().numpy(), aux["w"][c].cpu().numpy().astype(np.float64),
                Tx[c].cpu().numpy().astype(np.complex128), To, ao)
    else:
        n = xd.shape[1]
        left = O.pad_left(n_fft, framing)
        for c, f0, nf in frame_slices:
            # global frame f reads samples [f*hop - left, f*hop - left + n_fft).  The slice starts on a frame
            # boundary a = g0*hop, so slice frame j IS global frame g0 + j; frames f0 .. f0+nf-1 lie inside the slice
            # (or touch the true ends of the recording, where the slice's padding is the recording's padding)
            g0 = max(0, (f0 * hop - left) // hop)
            a = g0 * hop
            b = min(n, (f0 + nf - 1) * hop - left + n_fft)
            assert a == 0 or a <= f0 * hop - left
            xs = xd[c, a:b].cpu().numpy().astype(np.float64)
            To, _, ao = O.ssq_stft(xs, win, **okw)
            sel = np.arange(f0 - g0, min(f0 - g0 + nf, To.shape[1]))
            gsel = g0 + sel
            aos = {k: (v[:, sel] if getattr(v, "ndim", 0) == 2 else v) for k, v in ao.items()}
            gi = torch.as_tensor(gsel, device=xd.device)
            one(aux["kb"][c][:, gi].cpu().numpy(), aux["w"][c][:, gi].cpu().numpy().astype(np.float64),
                Tx[c][:, gi].cpu().numpy().astype(np.complex128), To[:, sel], aos)
    total["kernel"] = name
    return total



@pytest.mark.parametrize("hop,N", [(32, 20000), (17, 5000), (64, 9000), (1, 700), (32, 100)])
def test_fast_path_512(hop, N):
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    x = np.random.default_rng(hop).standard_normal(N) * 30.0
    win = np.hanning(512)
    check_ssq(x, win, 512, hop, 30000.0, expect_kernel="h32r")
    Sx, _ = rs.stft(x, 512, hop, win, "reflect")
    assert "512" in _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, 512, hop, win, "reflect")
    assert rel(Sx, So) < RTOL
    for kw in (dict(padtype="zero"), dict(squeezing="lebesgue"), dict(gamma=40.0)):
        check_ssq(x, win, 512, hop, 30000.0, expect_kernel="h32r", **kw)



@pytest.mark.parametrize("hop,N", [(256, 40000), (100, 9000), (1024, 30000), (1, 1500), (32, 300)])
def test_fast_path_1024(hop, N):
    """n_fft=1024 register-FFT kernel (tests/stft_ssq_test.py:166-167: the reference's multichannel script uses
    n_fft=1024, hop_length=256): ssq / stft, options, a tonal signal (collision path), modulated."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(hop)
    x = rng.standard_normal(N) * 30.0
    win = np.hanning(1024)
    fs = 30000.0
    check_ssq(x, win, 1024, hop, fs, expect_kernel="1024")
    Sx, _ = rs.stft(x, 1024, hop, win, "reflect")
    assert "1024" in _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, 1024, hop, win, "reflect")
    assert rel(Sx, So) < RTOL
    for kw in (dict(padtype="zero"), dict(squeezing="lebesgue"), dict(gamma=40.0), dict(modulated=True)):
        check_ssq(x, win, 1024, hop, fs, expect_kernel="1024", **kw)
    # tonal: every bin of a frame is squeezed into a few destination bins (collision path)
    t = np.arange(N) / fs
    xt = np.sin(2 * np.pi * 1234.5 * t) + 0.3 * np.sin(2 * np.pi * 5000.0 * t)
    check_ssq(xt, win, 1024, hop, fs, expect_kernel="1024")
    Tx, _ = rs.ssq_stft(xt, win, n_fft=1024, hop_len=hop, fs=fs)
    Tx2, _ = rs.ssq_stft(xt, win, n_fft=1024, hop_len=hop, fs=fs)
    assert np.array_equal(Tx, Tx2)  # run-to-run identical



@pytest.mark.parametrize("hop,N", [(64, 1000), (64, 40000), (17, 5000), (300, 30000), (1, 900), (8, 100)])
def test_fast_path_256(hop, N):
    """n_fft=256 register-FFT kernel, four frames per warp (README / tests/stft_test.py:137-151: n_fft=256, hop 64)."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(hop + 1)
    x = rng.standard_normal(N) * 30.0
    win = np.hanning(256)
    fs = 1000.0
    check_ssq(x, win, 256, hop, fs, expect_kernel="256")
    Sx, _ = rs.stft(x, 256, hop, win, "reflect")
    assert "256" in _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, 256, hop, win, "reflect")
    assert rel(Sx, So) < RTOL
    for kw in (dict(padtype="zero"), dict(squeezing="lebesgue"), dict(gamma=40.0), dict(modulated=True)):
        check_ssq(x, win, 256, hop, fs, expect_kernel="256", **kw)
    t = np.arange(N) / fs
    xt = np.sin(2 * np.pi * 100.0 * t) + 0.3 * np.sin(2 * np.pi * 333.3 * t)  # README sine plus one
    check_ssq(xt, win, 256, hop, fs, expect_kernel="256")
    Tx, _ = rs.ssq_stft(xt, win, n_fft=256, hop_len=hop, fs=fs)
    Tx2, _ = rs.ssq_stft(xt, win, n_fft=256, hop_len=hop, fs=fs)
    assert np.array_equal(Tx, Tx2)


def test_fast_path_256_batched_matches_generic():
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    rng = np.random.default_rng(12)
    ch, n = 9, 33333
    x = torch.from_numpy((rng.standard_normal((ch, n)) * 10).astype(np.float32)).cuda()
    win = np.hanning(256)
    a = eng.ssq_stft(x, win, n_fft=256, hop_len=64, fs=1000.0).cpu().numpy()
    assert "256" in eng.last_kernel_name()
    eng.ctx.set_option("no_r256", 1)
    try:
        b = eng.ssq_stft(x, win, n_fft=256, hop_len=64, fs=1000.0).cpu().numpy()
        assert "generic" in eng.last_kernel_name()
    finally:
        eng.ctx.set_option("no_r256", 0)
    for c in range(ch):
        _flip_tolerant_compare(a[c].astype(np.complex128), b[c].astype(np.complex128), max_bad_frac=4e-3)


def test_fast_path_1024_batched_matches_generic():
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    rng = np.random.default_rng(11)
    ch, n = 7, 70001
    x = torch.from_numpy((rng.standard_normal((ch, n)) * 10).astype(np.float32)).cuda()
    win = np.hanning(1024)
    a = eng.ssq_stft(x, win, n_fft=1024, hop_len=256, fs=1000.0).cpu().numpy()
    assert "1024" in eng.last_kernel_name()
    eng.ctx.set_option("no_r1024", 1)
    try:
        b = eng.ssq_stft(x, win, n_fft=1024, hop_len=256, fs=1000.0).cpu().numpy()
        assert "generic" in eng.last_kernel_name()
    finally:
        eng.ctx.set_option("no_r1024", 0)
    for c in range(ch):
        _flip_tolerant_compare(a[c].astype(np.complex128), b[c].astype(np.complex128), max_bad_frac=4e-3)


def test_batched_device_api_matches_per_channel():
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    rng = np.random.default_rng(3)
    ch, n = 5, 12345
    x = rng.standard_normal((ch, n)).astype(np.float32) * 10
    win = np.hanning(512)
    xd = torch.from_numpy(x).cuda()
    Tx = eng.ssq_stft(xd, win, n_fft=512, hop_len=32, fs=30000.0)
    torch.cuda.synchronize()
    assert eng.last_kernel_name().startswith("ssq_stft512")
    Tx = Tx.cpu().numpy()
    assert Tx.shape == (ch, 257, (n - 1) // 32 + 1)
    rep = check_ssq_device(eng, xd, win, 512, 32, 30000.0, channels=(0, 4), expect_kernel="h32r")
    assert rep["unexplained"] == 0
    # strided rows + generic kernel (n_fft=256), then round trip through istft
    big = torch.zeros((ch, n + 100), dtype=torch.float32, device="cuda")
    big[:, :n] = xd
    Sx = eng.stft(big[:, :n], np.hanning(256), 256, 64)
    xr = eng.istft(Sx, np.hanning(256), 256, 64, N=n)
    torch.cuda.synchronize()
    assert float((xr - xd).abs().max()) < 2e-4 * float(xd.abs().max())
    # host-buffer entry point == device entry point
    out = np.empty((ch, 257, (n - 1) // 32 + 1), dtype=np.complex64)
    eng.ssq_stft_host(x.ctypes.data, ch, n, win, 512, 32, 30000.0, out.ctypes.data)
    assert np.array_equal(out, Tx)



def test_full_size_properties_config2_slice():
    """BASELINE config 2 geometry (1.8 M samples/channel, the benchmarked kernel) on a 4-channel cut of the bench's
    own synthetic recipe: every bin against the oracle (unexplained == 0 over 4 x 14.46 M bins), plus the
    size-independent properties -- linearity in x and flip-invariant column sums equal to dw * sum_k Sx[k]."""
    import torch
    import bench
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    ch, n = 4, 1_800_000
    x = bench.make_neural(torch, ch, n, 30000.0, torch.device("cuda", 0), 0x5351)
    win = np.hanning(512)
    fs = 30000.0
    rep = check_ssq_device(eng, x, win, 512, 32, fs, expect_kernel="h32r")
    assert rep["bins_total"] == 4 * 257 * 56250 and rep["unexplained"] == 0, rep
    Tx = eng.ssq_stft(x, win, 512, 32, fs)
    Sx = eng.stft(x, win, 512, 32)
    torch.cuda.synchronize()
    assert Tx.shape == (ch, 257, 56250)
    dw = 0.5 * fs / 256
    cs_T = Tx.sum(dim=1)
    cs_S = Sx.sum(dim=1) * dw
    scale = float(Sx.abs().max()) * dw
    assert float((cs_T - cs_S).abs().max()) < 5e-4 * scale * 16
    # scaling x by 2 scales Tx by 2 with identical bins (power-of-two scale is exact in fp32)
    Tx2 = eng.ssq_stft(x * 2, win, 512, 32, fs)
    torch.cuda.synchronize()
    assert torch.equal(Tx2, Tx * 2)


@pytest.mark.parametrize("N,wexp", [(20000, 1), (5000, 0), (777, 2), (100, 1), (4096 + 33, 1)])
def test_istft_fast_path_512_32(N, wexp):
    """n_fft=512 / hop=32 register overlap-add kernel against the oracle (irfft + OLA), on a
    MODIFIED spectrum with non-zero imaginary DC / Nyquist parts (irfft ignores them)."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(N + wexp)
    x = rng.standard_normal(N) * 7.0
    win = np.hanning(514)[1:-1].copy()
    So, _ = O.stft(x, 512, 32, win, "reflect")
    So = So * (1 + 0.1 * rng.standard_normal(So.shape)) + 0.05j * rng.standard_normal(So.shape)
    xr = rs.istft(So, win, n_fft=512, hop_len=32, N=N, win_exp=wexp)
    assert "istft512" in _lib.default_context().last_kernel_name()
    xo = O.istft(So, win, n_fft=512, hop_len=32, N=N, win_exp=wexp)
    assert np.abs(xr - xo).max() < RTOL * np.abs(xo).max()
    # fewer columns than the padded length allows, and more (extra columns are ignored: _stft.py:236)
    for cols in (So.shape[1] - 3, So.shape[1]):
        if cols < 1:
            continue
        S2 = np.ascontiguousarray(So[:, :cols])
        xr = rs.istft(S2, win, n_fft=512, hop_len=32, N=N, win_exp=wexp)
        xo = O.istft(S2, win, n_fft=512, hop_len=32, N=N, win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30)


def test_istft_batched_roundtrip_fast_path():
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    x = torch.randn((37, 30001), generator=g, device="cuda") * 3
    win = np.hanning(514)[1:-1].copy()
    Sx = eng.stft(x, win, 512, 32)
    xr = eng.istft(Sx, win, 512, 32, N=x.shape[1])
    torch.cuda.synchronize()
    assert eng.last_kernel_name().startswith("istft512")
    assert float((xr - x).abs().max()) < 2e-5 * float(x.abs().max())



def test_fast_kernels_agree_and_are_deterministic():
    """The n_fft=512/hop=32 register kernel against the generic shared-memory kernel (an independent
    implementation: radix-4 Stockham in shared memory, ascending-k accumulation) on collision-heavy input (tone +
    weak noise: most bins of a frame map to one destination) and on noise: run-to-run identical, equal across kernels
    up to the order of additions inside a bin, and every bin of both explained against the oracle."""
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    g = torch.Generator(device="cuda")
    g.manual_seed(9)
    n = 200_000
    t = torch.arange(n, device="cuda", dtype=torch.float64) / 30000.0
    tone = torch.sin(2 * np.pi * 1000.0 * t).to(torch.float32)
    x = torch.stack([tone * 50 + torch.randn(n, generator=g, device="cuda") * a for a in (0.0, 1e-3, 1.0, 30.0)])
    win = np.hanning(512)
    outs = {}
    try:
        for name, opt in (("h32r", 0), ("generic", 1)):
            eng.ctx.set_option("no_h32r", opt)
            a = eng.ssq_stft(x, win, 512, 32, 30000.0)
            b = eng.ssq_stft(x, win, 512, 32, 30000.0)
            torch.cuda.synchronize()
            assert torch.equal(a, b), name
            outs[name] = (a, eng.last_kernel_name())
            rep = check_ssq_device(eng, x[:, :60_000].contiguous(), win, 512, 32, 30000.0)
            assert rep["unexplained"] == 0, (name, rep)
    finally:
        eng.ctx.set_option("no_h32r", 0)
    assert "h32r" in outs["h32r"][1] and "generic" in outs["generic"][1]
    ref = outs["generic"][0]
    sc = float(ref.abs().max())
    d = (outs["h32r"][0] - ref).abs()
    # identical bins -> only rounding differences; edge flips (classified above) are few
    assert float((d > 1e-4 * sc).float().mean()) < 1e-3
    assert float((outs["h32r"][0].sum(dim=1) - ref.sum(dim=1)).abs().max()) < 2e-3 * sc


def test_context_options_are_set_only_through_set_option(monkeypatch):
    """The context has five options; the names of the removed CTA-shape / CWT tuning switches are unknown
    (ValueError); and nothing is read from the environment: SSQ_NO_H32R=1 leaves a new context on the n_fft 512
    register kernel."""
    import torch
    from ssqueeze_rs_b200._lib import Context
    from ssqueeze_rs_b200.batch import Engine
    ctx = Context(0)
    for name in ("no_h32r", "no_r1024", "no_r256", "no_cwt_fused", "upstream_framing"):
        ctx.set_option(name, 1)
        ctx.set_option(name, 0)
    for name in ("h32r_nw", "istft_nw", "fft128_tc", "cwt_fused_tc", "no_fft128", "no_cwt_prune", "cwt_ws_mb"):
        with pytest.raises(ValueError):
            ctx.set_option(name, 1)
    monkeypatch.setenv("SSQ_NO_H32R", "1")
    eng = Engine(0)
    x = torch.randn((2, 5000), device="cuda")
    eng.ssq_stft(x, np.hanning(512), 512, 32, 30000.0)
    torch.cuda.synchronize()
    assert "h32r" in eng.last_kernel_name()



def test_long_recording_config5_geometry():
    """BASELINE config 5 geometry (10 min @ 30 kHz = 18 M samples per channel, 562 500 frames) on a
    2-channel cut: 64-bit indexing, slices of frames at the start, far into and at the end of the recording against
    the oracle with every bin classified (a frame only depends on its own 512 samples, so the oracle runs on the
    samples of the slice), and the column-sum property."""
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    g = torch.Generator(device="cuda")
    g.manual_seed(11)
    ch, n = 2, 18_000_000
    x = torch.randn((ch, n), generator=g, device="cuda") * 15
    win = np.hanning(512)
    fs = 30000.0
    # slices start where (a + left) is a multiple of hop: f0*hop - left -> choose f0 >= 8
    rep = check_ssq_device(eng, x, win, 512, 32, fs, expect_kernel="h32r",
                           frame_slices=[(0, 0, 96), (1, 280_000, 128), (0, 431_111, 64), (1, 562_500 - 96, 96)])
    assert rep["unexplained"] == 0 and rep["bins_total"] >= 257 * 300, rep
    Tx = eng.ssq_stft(x, win, 512, 32, fs)
    assert Tx.shape == (ch, 257, 562_500)
    Sx = eng.stft(x[1:2], win, 512, 32)
    torch.cuda.synchronize()
    dw = 0.5 * fs / 256
    d = (Tx[1].sum(dim=0) - Sx[0].sum(dim=0) * dw).abs().max()
    assert float(d) < 8e-3 * float(Sx.abs().max()) * dw


def test_channel_sharder_matches_engine():
    """Host-side multi-device path (one context + host thread per device, host gather only);
    with one GPU the two 'devices' are two contexts on cuda:0."""
    import torch
    from ssqueeze_rs_b200.batch import ChannelSharder, Engine
    rng = np.random.default_rng(21)
    x = (rng.standard_normal((7, 20000)) * 5).astype(np.float32)
    win = np.hanning(512)
    ref = Engine(0).ssq_stft(torch.from_numpy(x).cuda(), win, 512, 32, 30000.0).cpu().numpy()
    for devs in ([0], [0, 0], [0, 0, 0]):
        out = ChannelSharder(devs).ssq_stft(x, win, 512, 32, 30000.0)
        assert out.shape == ref.shape and np.array_equal(out, ref)


@pytest.mark.parametrize("hop,N", [(1, 900), (17, 5000), (64, 9000), (128, 20000), (256, 7000), (600, 10000)])
def test_istft_512_any_hop(hop, N):
    """The n_fft=512 tile kernel at hops other than 32 (gather overlap-add with a runtime hop)."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(hop)
    x = rng.standard_normal(N)
    win = np.hanning(514)[1:-1].copy()
    So, _ = O.stft(x, 512, hop, win, "reflect")
    So = So * (1 + 0.05 * rng.standard_normal(So.shape))
    for wexp in (1, 0):
        xr = rs.istft(So, win, n_fft=512, hop_len=hop, N=N, win_exp=wexp)
        assert "istft512_" in _lib.default_context().last_kernel_name()
        xo = O.istft(So, win, n_fft=512, hop_len=hop, N=N, win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30), (hop, wexp)


def test_modulated_fast_path_and_issq_roundtrip_512():
    """`modulated=True` (Sx[k] (-1)^k before squeezing) on the n_fft=512 fast kernel, hop 1 and 32, and the
    issq_stft round trip (old/tests/reconstruction_test.py:182-206: MAE < 0.1) at n_fft=512."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    x = np.random.default_rng(77).standard_normal(1500)
    win = np.hanning(514)[1:-1].copy()
    for hop in (1, 32):
        check_ssq(x, win, 512, hop, 250.0, modulated=True, expect_kernel="h32r")
    Tx, _ = rs.ssq_stft(x, win, n_fft=512, hop_len=1, fs=250.0, modulated=True)
    y = rs.issq_stft(Tx, win, n_fft=512, hop_len=1, fs=250.0)
    sh = 512 // 2 - (512 - 1) // 2
    assert np.abs(y[:len(x) - sh] - x[sh:]).mean() < 0.1


def test_fast_kernels_randomised_sweep():
    """Seeded sweep over the three register-FFT kernels (n_fft 256 / 512 / 1024): random lengths (including shorter
    than n_fft and lengths that leave ragged tiles), hops, window families and lengths (win_len < n_fft is centre
    padded, ssq_stft.rs:104-119), padding, squeezing, gamma, modulation -- each against the float64 oracle."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(20261018)
    wins = {"hann": np.hanning, "hamming": np.hamming, "blackman": np.blackman,
            "rand": lambda m: 0.2 + rng.random(m)}
    for case in range(36):
        n_fft = (256, 512, 1024)[case % 3]
        N = int(rng.choice([rng.integers(1, n_fft), rng.integers(n_fft, 6 * n_fft), rng.integers(6 * n_fft, 40 * n_fft)]))
        hop = int(rng.choice([1, 2, 31, 32, 33, 64, 100, 256, n_fft, n_fft + 17])) if N > 2000 else int(rng.integers(1, 70))
        if N // hop > 6000:
            hop = max(hop, N // 6000)
        wname = list(wins)[case % 4]
        win_len = n_fft if case % 5 else int(rng.integers(n_fft // 4, n_fft))
        win = np.asarray(wins[wname](win_len), dtype=np.float64)
        kw = dict(padtype=("reflect", "zero")[case % 2], squeezing=("sum", "lebesgue")[(case // 2) % 2 if case % 7 == 0 else 0],
                  gamma=(None, 1e-3, 5.0)[case % 3 if case % 4 == 0 else 0], modulated=bool(case % 6 == 5))
        fs = float(rng.choice([1.0, 1000.0, 30000.0]))
        x = rng.standard_normal(N) * rng.choice([1e-3, 1.0, 300.0])
        if case % 9 == 4:
            x += 5.0 * np.abs(x).max() * np.sin(2 * np.pi * 0.123 * np.arange(N))
        try:
            rep = check_ssq(x, win, n_fft, hop, fs, expect_kernel=str(n_fft), **kw)
        except AssertionError as e:
            raise AssertionError((case, n_fft, N, hop, wname, kw, fs)) from e
        assert "generic" not in rep["kernel"], (case, rep)
        if win_len == n_fft:
            Sx, _ = rs.stft(x, n_fft, hop, win, kw["padtype"])
            So, _ = O.stft(x, n_fft, hop, win, kw["padtype"])
            assert rel(Sx, So) < RTOL, (case, n_fft, N, hop, wname)


@pytest.mark.parametrize("hop,N", [(256, 40000), (100, 9000), (1, 1500), (1024, 30000), (1500, 20000), (32, 300)])
def test_istft_1024(hop, N):
    """n_fft=1024 inverse (register 32 x 32 FFT, packed frame pairs, gather overlap-add) against the oracle, both
    window exponents, plus the round trip through the n_fft=1024 forward kernel."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(hop + 7)
    x = rng.standard_normal(N)
    win = np.hanning(1026)[1:-1].copy()
    So, _ = O.stft(x, 1024, hop, win, "reflect")
    So = So * (1 + 0.05 * rng.standard_normal(So.shape))
    for wexp in (1, 0):
        xr = rs.istft(So, win, n_fft=1024, hop_len=hop, N=N, win_exp=wexp)
        assert "istft1024" in _lib.default_context().last_kernel_name()
        xo = O.istft(So, win, n_fft=1024, hop_len=hop, N=N, win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30), (hop, wexp)
    if hop <= 512:
        Sx, _ = rs.stft(x, 1024, hop, win, "reflect")
        xb = rs.istft(Sx, win, n_fft=1024, hop_len=hop, N=N)
        assert np.abs(xb - x).max() < 1e-4 * np.abs(x).max(), hop


@pytest.mark.parametrize("hop,N", [(64, 40000), (17, 5000), (1, 900), (256, 30000), (300, 20000), (8, 100)])
def test_istft_256(hop, N):
    """n_fft=256 inverse (8 x 32 register FFT, four packed pairs of frames per warp) against the oracle, both window
    exponents, plus the round trip through the n_fft=256 forward kernel."""
    rs = _rs()
    from ssqueeze_rs_b200 import _lib
    rng = np.random.default_rng(hop + 11)
    x = rng.standard_normal(N)
    win = np.hanning(258)[1:-1].copy()
    So, _ = O.stft(x, 256, hop, win, "reflect")
    So = So * (1 + 0.05 * rng.standard_normal(So.shape))
    for wexp in (1, 0):
        xr = rs.istft(So, win, n_fft=256, hop_len=hop, N=N, win_exp=wexp)
        assert "istft256" in _lib.default_context().last_kernel_name()
        xo = O.istft(So, win, n_fft=256, hop_len=hop, N=N, win_exp=wexp)
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30), (hop, wexp)
    if hop <= 128:
        Sx, _ = rs.stft(x, 256, hop, win, "reflect")
        xb = rs.istft(Sx, win, n_fft=256, hop_len=hop, N=N)
        assert np.abs(xb - x).max() < 1e-4 * np.abs(x).max(), hop


def test_rs_ssq_stft_batch_equals_the_per_channel_drop_in():
    """`_rs.ssq_stft_batch` (all channels in one call, complex64 in pinned host memory or on the device) against the
    reference-shaped scalar call in the loop of tests/stft_ssq_test.py:230-251: same kernel, same bits."""
    import torch
    from ssqueeze_rs_b200 import _rs
    rng = np.random.default_rng(5)
    x = rng.standard_normal((5, 20000)) * 10
    win = np.hanning(512)
    Tx, sf = _rs.ssq_stft_batch(x, win, n_fft=512, hop_len=32, fs=30000.0)
    assert Tx.dtype == np.complex64 and Tx.shape == (5, 257, 625)
    for c in range(5):
        Tc, sfc = _rs.ssq_stft(x[c], win, n_fft=512, hop_len=32, fs=30000.0)
        assert np.array_equal(sf, sfc)
        assert np.array_equal(Tx[c].astype(np.complex128), Tc)
    # the pinned result is reusable as `out=`; float32 input; options pass through
    x32 = x.astype(np.float32)
    Tx2, _ = _rs.ssq_stft_batch(x32, win, n_fft=512, hop_len=32, fs=30000.0, out=Tx, modulated=True, padtype="zero")
    assert Tx2 is Tx
    Tm, _ = _rs.ssq_stft(x32[3].astype(np.float64), win, n_fft=512, hop_len=32, fs=30000.0, modulated=True, padtype="zero")
    assert np.array_equal(Tx[3].astype(np.complex128), Tm)
    # Tx kept on the device
    Td, _ = _rs.ssq_stft_batch(x, win, n_fft=512, hop_len=32, fs=30000.0, device_out=True)
    assert isinstance(Td, torch.Tensor) and Td.is_cuda
    T0, _ = _rs.ssq_stft_batch(x, win, n_fft=512, hop_len=32, fs=30000.0)
    assert np.array_equal(Td.cpu().numpy(), T0)


@pytest.mark.parametrize("n,n_fft,hop", [(300, 512, 32), (5000, 500, 7), (4097, 256, 64), (9000, 8192, 1000), (64, 16, 1)])
def test_rs_ssq_stft_batch_odd_geometries(n, n_fft, hop):
    """The batched drop-in through every kernel family (signal shorter than the frame, Bluestein lengths, the rows path
    above 4096 points, tiny frames at hop 1): equal to the scalar drop-in channel by channel."""
    from ssqueeze_rs_b200 import _rs
    rng = np.random.default_rng(n + n_fft)
    x = rng.standard_normal((3, n))
    win = np.hanning(n_fft)
    Tx, sf = _rs.ssq_stft_batch(x, win, n_fft=n_fft, hop_len=hop, fs=1000.0)
    for c in range(3):
        Tc, sfc = _rs.ssq_stft(x[c], win, n_fft=n_fft, hop_len=hop, fs=1000.0)
        assert Tx[c].shape == Tc.shape and np.array_equal(sf, sfc)
        assert np.array_equal(Tx[c].astype(np.complex128), Tc), (n, n_fft, hop, c)


@pytest.mark.parametrize("n,n_fft,hop", [(20000, 512, 32), (20000, 1024, 256), (5000, 500, 7), (300, 128, 1)])
def test_rs_stft_batch_equals_the_per_channel_drop_in(n, n_fft, hop):
    """`_rs.stft_batch` (host pipeline of ssq_stft_host_f32 / Tx on the device) against the scalar `_rs.stft` loop."""
    from ssqueeze_rs_b200 import _rs
    rng = np.random.default_rng(n_fft + hop)
    x = rng.standard_normal((4, n)) * 10
    win = np.hanning(n_fft)
    Sx, fr = _rs.stft_batch(x, n_fft, hop, win, "reflect")
    assert Sx.dtype == np.complex64
    for c in range(4):
        Sc, frc = _rs.stft(x[c], n_fft, hop, win, "reflect")
        assert np.array_equal(fr, frc)
        assert np.array_equal(Sx[c].astype(np.complex128), Sc), (n, n_fft, hop, c)
    Sd, _ = _rs.stft_batch(x, n_fft, hop, win, "reflect", device_out=True)
    assert np.array_equal(Sd.cpu().numpy(), Sx)
    Sz, _ = _rs.stft_batch(x.astype(np.float32), n_fft, hop, win, "zero", out=Sx)
    assert Sz is Sx

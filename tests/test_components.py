"""Component (curve-band) inversion of issq_cwt and issq_stft (old/ssqueezepy/_ssq_cwt.py:380-402) on the device, for a
batch of channels: `Engine.issq_cwt` / `Engine.issq_stft` with `cc`, `cw`, `_rs.issq_stft(..., cc=, cw=)` and
`compat.issq_stft(..., cc, cw)`, all through `issq_components_kernel`.

The float64 reference of the STFT side is `stft_components` below: the oracle's `invert_components` (pinned to upstream's
`_invert_components` by upstream_components.npz) times the factor 2 / (w[n_fft // 2] fs) that upstream applies after
either branch of issq_stft (pinned by k2_issq / k4_issq of upstream_compat.npz).  No upstream output of the STFT
component path itself is committed.

CPU: that reference against upstream's full inverse; argument errors before any device work.  GPU: adversarial bands
against the reference, the upstream golden through the batch entry, bit-equalities between the entry points, compat,
and ssq_cwt / ssq_stft -> extract_ridges -> component inversion end to end on the device."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import ssq_oracle as O

G = os.path.join(os.path.dirname(__file__), "golden")
I32_MAX, I32_MIN = 2**31 - 1, -2**31
SSQ_EINVAL, SSQ_EUNSUPPORTED = 1, 4


def stft_components(Tx, window, n_fft, fs, cc, cw):
    """float64 reference of issq_stft with curve bands: invert_components(Tx, cc, cw) * 2 / w[n_fft // 2] / fs."""
    wsz = O.fit_window(window, n_fft)
    return O.invert_components(Tx, cc, cw) * (2.0 / wsz[n_fft // 2]) / fs


def cwt_components(Tx, wavelet, scales, cc, cw):
    return O.issq_cwt(Tx, wavelet, scales, cc, cw)


def _compat_cases():
    z = np.load(os.path.join(G, "upstream_compat.npz"))
    for ci in range(len(z["cases"])):
        p = f"k{ci}_"
        if p + "issq" in z.files:
            yield dict(Tx=z[p + "Tx"], window_fit=z[p + "window_fit"], issq=z[p + "issq"], n_fft=len(z[p + "window_fit"]),
                       wk=int(z["cases"][ci][4]))


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_stft_reference_against_upstream_full_inverse():
    """One band covering every row is upstream's full issq_stft (k2_issq, k4_issq) with a zero residual; disjoint bands
    plus the residual sum to the same values."""
    n = 0
    for c in _compat_cases():
        Tx, w, nf = c["Tx"], c["window_fit"], c["n_fft"]
        rows, cols = Tx.shape
        ref = c["issq"]
        tol = 1e-12 * np.abs(ref).max()
        y = stft_components(Tx, w, nf, 1.0, np.zeros(cols, np.int32), np.full(cols, rows, np.int32))
        assert y.shape == (2, cols)
        assert np.abs(y[0] - ref).max() <= tol and np.all(y[1] == 0.0)
        assert np.abs(O.issq_stft(Tx, w, nf) - ref).max() <= tol
        cc = np.tile(np.array([5, 20, rows - 2], np.int32), (cols, 1))
        cw = np.tile(np.array([5, 8, 1], np.int32), (cols, 1))  # rows 0..10, 12..28, the last three; residual 11, 29..
        y = stft_components(Tx, w, nf, 1.0, cc, cw)
        assert y.shape == (4, cols) and np.abs(y[3]).max() > 0.0
        assert np.abs(y.sum(0) - ref).max() <= tol
        n += 1
    assert n == 2


def test_argument_errors_before_any_device_work(built_lib):
    from ssqueeze_rs_b200 import _rs, compat
    rng = np.random.default_rng(0)
    Tx = (rng.standard_normal((33, 50)) + 1j * rng.standard_normal((33, 50))).astype(np.complex128)
    w = np.hanning(64)
    cc = np.zeros((50, 2), np.int32)
    for fn in (lambda **k: _rs.issq_stft(Tx, w, **k), lambda **k: compat.issq_stft(Tx, w, **k)):
        with pytest.raises(ValueError, match="go together"):
            fn(cc=cc)
        with pytest.raises(ValueError, match="go together"):
            fn(cw=cc)
        with pytest.raises(ValueError):
            fn(cc=cc, cw=np.zeros((50, 3), np.int32))
        with pytest.raises(ValueError):
            fn(cc=np.zeros(49, np.int32), cw=np.zeros(49, np.int32))


def test_abi_component_count_and_context_checks(built_lib):
    """K outside 1..16 is SSQ_EUNSUPPORTED before the context is looked at; then a NULL context is SSQ_EINVAL."""
    lib = built_lib
    buf = np.zeros(4096, np.float64)
    p = C.c_void_p(buf.ctypes.data)
    w = np.hanning(64)
    wp = C.c_void_p(w.ctypes.data)
    sc = np.array([1.0, 2.0])
    sp = C.c_void_p(sc.ctypes.data)
    calls = {
        "cwt batch": lambda K: lib.ssq_issq_cwt_components_batch_f32(None, p, 1, 2, 10, 0, sp, p, p, K, p),
        "stft batch": lambda K: lib.ssq_issq_stft_components_batch_f32(None, p, 1, 33, 10, wp, 64, 64, 1.0, p, p, K, p),
        "stft f64": lambda K: lib.ssq_issq_stft_components_f64(None, p, 33, 10, wp, 64, 64, 1, 1.0, p, p, K, p),
    }
    for name, call in calls.items():
        for K in (0, 17, -1):
            assert call(K) == SSQ_EUNSUPPORTED, (name, K)
            assert b"components" in lib.ssq_last_error(None), name
        for K in (1, 16):
            assert call(K) == SSQ_EINVAL, (name, K)
            assert lib.ssq_last_error(None) == b"ctx is NULL", name


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
def _engine():
    from ssqueeze_rs_b200.batch import Engine
    return Engine(0)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _random_tx(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def _adversarial_bands(rng, shape, n_rows):
    """cc / cw int32 of `shape` mixing ordinary bands with cc = -1, -5, >= n_rows, INT32_MAX and cw = 0, < 0, > n_rows,
    INT32_MAX, INT32_MIN: everything the clipping rule has to get right, overlaps included."""
    cc = rng.integers(0, n_rows, size=shape)
    cw = rng.integers(0, 5, size=shape)
    pick = rng.integers(0, 10, size=shape)
    cc[pick == 0] = -1
    cc[pick == 1] = -5
    cc[pick == 2] = n_rows + rng.integers(0, 3, size=int((pick == 2).sum()))
    cc[pick == 3] = I32_MAX
    pick = rng.integers(0, 10, size=shape)
    cw[pick == 0] = 0
    cw[pick == 1] = -rng.integers(1, 4, size=int((pick == 1).sum()))
    cw[pick == 2] = n_rows + 7
    cw[pick == 3] = I32_MAX
    cw[pick == 4] = I32_MIN
    return cc.astype(np.int32), cw.astype(np.int32)


def _close_per_row(got, ref, rtol=1e-5):
    """|got - ref| <= rtol * max |ref| of each output row (exactly 0 where a row of the reference is 0)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape
    lim = rtol * np.abs(ref).max(axis=-1, keepdims=True)
    bad = np.abs(got - ref) > lim
    assert not bad.any(), (int(bad.sum()), float(np.abs(got - ref).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3, 16])
def test_adversarial_bands_against_the_reference(K):
    """CWT and STFT, batch and float64 entries: every channel and row against invert_components x the factor."""
    from ssqueeze_rs_b200 import _rs
    eng = _engine()
    rng = np.random.default_rng(100 + K)
    ch, n = 3, 1000
    # CWT: 37 rows (the unrolled row loop plus a tail), ascending scales
    sc = 2.0 ** np.linspace(1, 6, 37)
    Tx = _random_tx(rng, (ch, 37, n))
    cc, cw = _adversarial_bands(rng, (ch, n, K), 37)
    for wav in ("gmw", "morlet"):
        x = eng.issq_cwt(_dev(Tx), sc, wav, cc=_dev(cc), cw=_dev(cw))
        assert eng.last_kernel_name() == "issq_components_kernel"
        assert x.shape == (ch, K + 1, n)
        x = x.cpu().numpy()
        for c in range(ch):
            ref = cwt_components(Tx[c].astype(np.complex128), wav, sc, cc[c], cw[c])
            _close_per_row(x[c], ref)
        x1 = _rs.issq_cwt(Tx[1].astype(np.complex128), wav, sc, cc[1], cw[1])
        assert _rs._lib.default_context().last_kernel_name() == "issq_components_kernel"
        _close_per_row(x1, cwt_components(Tx[1].astype(np.complex128), wav, sc, cc[1], cw[1]))
    # STFT: n_fft 64 -> 33 rows
    win, nf, fs = np.hanning(64), 64, 3.0
    Tx = _random_tx(rng, (ch, 33, n))
    cc, cw = _adversarial_bands(rng, (ch, n, K), 33)
    y = eng.issq_stft(_dev(Tx), win, nf, fs, cc=_dev(cc), cw=_dev(cw))
    assert eng.last_kernel_name() == "issq_components_kernel"
    assert y.shape == (ch, K + 1, n)
    y = y.cpu().numpy()
    for c in range(ch):
        _close_per_row(y[c], stft_components(Tx[c].astype(np.complex128), win, nf, fs, cc[c], cw[c]))
    y1 = _rs.issq_stft(Tx[2].astype(np.complex128), win, nf, fs=fs, cc=cc[2], cw=cw[2])
    assert _rs._lib.default_context().last_kernel_name() == "issq_components_kernel"
    assert y1.shape == (K + 1, n)
    _close_per_row(y1, stft_components(Tx[2].astype(np.complex128), win, nf, fs, cc[2], cw[2]))


@pytest.mark.gpu
def test_upstream_golden_through_the_batch_entry():
    """upstream_components.npz (upstream's own `_invert_components`) through `Engine.issq_cwt`, up to the factor."""
    z = np.load(os.path.join(G, "upstream_components.npz"))
    Tx, cc, cw = z["Tx"], z["cc"], z["cw"]
    sc = 2.0 ** np.linspace(1, 5, Tx.shape[0])
    eng = _engine()
    for wav in ("gmw", "morlet"):
        x = eng.issq_cwt(_dev(Tx.astype(np.complex64)[None]), sc, wav, cc=_dev(cc[None]), cw=_dev(cw[None]))
        assert eng.last_kernel_name() == "issq_components_kernel"
        x = x[0].cpu().numpy().astype(np.float64)
        f = (2.0 / O.adm_ssq(wav)) * np.log(sc[1] / sc[0])
        assert x.shape == (4, 300)
        assert np.abs(x / f - z["x"]).max() < 1e-4 * np.abs(z["x"]).max(), wav


@pytest.mark.gpu
def test_one_path_same_bits():
    """The float64 entries run the batch entry's kernel on the fp32-rounded Tx: the same bits.  Channel c of a batch is
    the one-channel call; two runs agree; a band over every row is the full inversion (CWT: bit for bit; STFT: within
    the reordering bound of issq_stft_kernel's two accumulators)."""
    import torch
    from ssqueeze_rs_b200 import _rs
    eng = _engine()
    rng = np.random.default_rng(7)
    ch, ns, n, K = 5, 45, 3001, 3
    sc = 2.0 ** np.linspace(0.5, 7, ns)
    Tx = _random_tx(rng, (ch, ns, n))
    cc, cw = _adversarial_bands(rng, (ch, n, K), ns)
    dTx, dcc, dcw = _dev(Tx), _dev(cc), _dev(cw)
    x = eng.issq_cwt(dTx, sc, "gmw", cc=dcc, cw=dcw)
    x2 = eng.issq_cwt(dTx, sc, "gmw", cc=dcc, cw=dcw)
    assert eng.last_kernel_name() == "issq_components_kernel"
    assert torch.equal(x, x2)
    for c in range(ch):
        xc = eng.issq_cwt(dTx[c:c + 1], sc, "gmw", cc=dcc[c:c + 1], cw=dcw[c:c + 1])
        assert torch.equal(xc[0], x[c]), c
    xh = _rs.issq_cwt(Tx[3].astype(np.complex128), "gmw", sc, cc[3], cw[3])
    assert np.array_equal(xh, x[3].cpu().numpy().astype(np.float64))
    # a band over every row (K = 1 as [channels, n], cw an int) is the full inversion, bit for bit; residual 0
    every = torch.zeros((ch, n), dtype=torch.int32, device="cuda")
    xa = eng.issq_cwt(dTx, sc, "gmw", cc=every, cw=ns)
    assert xa.shape == (ch, 2, n) and eng.last_kernel_name() == "issq_components_kernel"
    full = eng.issq_cwt(dTx, sc, "gmw")
    assert eng.last_kernel_name() == "icwt_kernel"
    assert torch.equal(xa[:, 0], full) and not xa[:, 1].any()

    # STFT
    win, nf, fs = np.hanning(128), 128, 2.0
    Tx = _random_tx(rng, (ch, 65, n))
    cc, cw = _adversarial_bands(rng, (ch, n, K), 65)
    dTx, dcc, dcw = _dev(Tx), _dev(cc), _dev(cw)
    y = eng.issq_stft(dTx, win, nf, fs, cc=dcc, cw=dcw)
    assert eng.last_kernel_name() == "issq_components_kernel"
    assert torch.equal(y, eng.issq_stft(dTx, win, nf, fs, cc=dcc, cw=dcw))
    for c in range(ch):
        assert torch.equal(eng.issq_stft(dTx[c:c + 1], win, nf, fs, cc=dcc[c:c + 1], cw=dcw[c:c + 1])[0], y[c]), c
    yh = _rs.issq_stft(Tx[1].astype(np.complex128), win, nf, fs=fs, cc=cc[1], cw=cw[1])
    assert np.array_equal(yh, y[1].cpu().numpy().astype(np.float64))
    ya = eng.issq_stft(dTx, win, nf, fs, cc=every, cw=65)
    full = eng.issq_stft(dTx, win, nf, fs)
    assert eng.last_kernel_name() == "issq_stft_kernel"
    assert not ya[:, 1].any()
    scale = 2.0 / (O.fit_window(win, nf)[nf // 2] * fs)
    bound = 65 * np.finfo(np.float32).eps * np.abs(Tx.real).sum(axis=1) * scale  # [ch, n]
    assert np.all(np.abs(ya[:, 0].cpu().numpy() - full.cpu().numpy()) <= bound)


@pytest.mark.gpu
def test_compat_components_on_the_upstream_maps():
    """compat.issq_stft(Tx, cc=, cw=) on upstream's own maps equals the reference; 1-D cc / cw are one band."""
    from ssqueeze_rs_b200 import compat
    rng = np.random.default_rng(3)
    n = 0
    for c in _compat_cases():
        Tx, nf = c["Tx"], c["n_fft"]
        rows, cols = Tx.shape
        window = np.hanning(nf + 2)[1:-1].copy() if c["wk"] == 0 else {1: "hann", 2: None, 3: "hamming"}[c["wk"]]
        cc, cw = _adversarial_bands(rng, (cols, 2), rows)
        y = compat.issq_stft(Tx, window=window, cc=cc, cw=cw, n_fft=nf)
        assert compat._context().last_kernel_name() == "issq_components_kernel"
        assert y.shape == (3, cols)
        Tr = Tx.astype(np.complex64).astype(np.complex128)
        _close_per_row(y, stft_components(Tr, c["window_fit"], nf, 1.0, cc, cw))
        # the whole map as one band: upstream's full inverse
        ya = compat.issq_stft(Tx, window=window, cc=np.zeros(cols, np.int32), cw=np.full(cols, rows), n_fft=nf)
        assert ya.shape == (2, cols)
        assert np.abs(ya[0] - c["issq"]).max() < 1e-5 * np.abs(c["issq"]).max()
        y1 = compat.issq_stft(Tx, window=window, cc=cc[:, 0], cw=cw[:, 0], n_fft=nf)
        assert y1.shape == (2, cols) and np.array_equal(y1[0], y[0])
        n += 1
    assert n == 2


def _two_sources(ch, n):
    """Per channel a tone and a linear chirp at channel-dependent frequencies (cycles per sample), well apart."""
    t = np.arange(n, dtype=np.float64)
    tones, chirps = [], []
    for c in range(ch):
        f0 = 0.02 + 0.005 * c
        g0, g1 = 0.10 + 0.01 * c, 0.22 + 0.01 * c
        tones.append(np.cos(2 * np.pi * f0 * t))
        chirps.append(0.8 * np.cos(2 * np.pi * (g0 * t + 0.5 * (g1 - g0) / n * t * t)))
    return np.array(tones), np.array(chirps)


def _check_separation(comp, tones, chirps, shift=0):
    """Each of the two components correlates above 0.9 with one clean source in the interior, and not the same one."""
    n = comp.shape[-1]
    core = slice(n // 8, n - n // 8)
    for c in range(comp.shape[0]):
        best = []
        for k in range(2):
            y = comp[c, k, core]
            r = [np.corrcoef(y, np.roll(s[c], -shift)[core])[0, 1] for s in (tones, chirps)]
            best.append(int(np.argmax(r)))
            assert max(r) > 0.9, (c, k, r)
        assert sorted(best) == [0, 1], (c, best)


@pytest.mark.gpu
def test_end_to_end_on_the_device():
    """ssq_cwt / ssq_stft -> extract_ridges -> component inversion, 4 channels x 2^15 samples, Tx and the ridge indices
    never leave the device; the components equal the reference on the device's own Tx and indices."""
    import torch
    eng = _engine()
    ch, n = 4, 1 << 15
    tones, chirps = _two_sources(ch, n)
    x = _dev((tones + chirps).astype(np.float32))
    # CWT
    sc = eng.default_scales(n, 16)
    Tx = eng.ssq_cwt(x, "gmw", sc, nv=16)
    idx = eng.extract_ridges(Tx, sc, penalty=2.0, n_ridges=2, bw=8, transform="cwt")
    comp = eng.issq_cwt(Tx, sc, "gmw", cc=idx, cw=8)
    assert eng.last_kernel_name() == "issq_components_kernel"
    assert comp.shape == (ch, 3, n)
    comp = comp.cpu().numpy()
    Th, ih = Tx.cpu().numpy(), idx.cpu().numpy()
    for c in range(ch):
        _close_per_row(comp[c], cwt_components(Th[c].astype(np.complex128), "gmw", sc, ih[c], np.full_like(ih[c], 8)))
    _check_separation(comp, tones, chirps)
    del Tx, Th
    torch.cuda.empty_cache()
    # STFT at hop 1, modulated
    win, nf = np.hanning(256), 256
    Tx = eng.ssq_stft(x, win, nf, 1, 1.0, modulated=True)
    sf = np.arange(nf // 2 + 1) * 0.5 / (nf // 2) + 1e-9
    idx = eng.extract_ridges(Tx, sf, penalty=0.5, n_ridges=2, bw=4, transform="stft")
    comp = eng.issq_stft(Tx, win, nf, 1.0, cc=idx, cw=4)
    assert eng.last_kernel_name() == "issq_components_kernel"
    assert comp.shape == (ch, 3, n)
    comp = comp.cpu().numpy()
    Th, ih = Tx.cpu().numpy(), idx.cpu().numpy()
    for c in range(ch):
        _close_per_row(comp[c], stft_components(Th[c].astype(np.complex128), win, nf, 1.0, ih[c], np.full_like(ih[c], 4)))
    # y[j] estimates x[j + n_fft // 2 - (n_fft - 1) // 2] in the crate's framing
    _check_separation(comp, tones, chirps, shift=nf // 2 - (nf - 1) // 2)


@pytest.mark.gpu
def test_engine_argument_errors():
    import torch
    eng = _engine()
    Tx = torch.zeros((2, 33, 40), dtype=torch.complex64, device="cuda")
    cc = torch.zeros((2, 40, 3), dtype=torch.int32, device="cuda")
    sc = 2.0 ** np.linspace(1, 4, 33)
    w = np.hanning(64)
    for call in (lambda **k: eng.issq_cwt(Tx, sc, **k), lambda **k: eng.issq_stft(Tx, w, 64, **k)):
        with pytest.raises(ValueError, match="go together"):
            call(cc=cc)
        with pytest.raises(ValueError, match="go together"):
            call(cw=3)
        with pytest.raises(ValueError):
            call(cc=cc, cw=cc[:, :, :2])
        with pytest.raises(ValueError):
            call(cc=cc[:, :39], cw=1)
        with pytest.raises(ValueError):
            call(cc=cc.long(), cw=1)
        with pytest.raises(ValueError):
            call(cc=cc.cpu(), cw=1)
    from ssqueeze_rs_b200 import SsqError
    with pytest.raises(SsqError, match="components"):
        eng.issq_cwt(Tx, sc, cc=torch.zeros((2, 40, 17), dtype=torch.int32, device="cuda"), cw=1)

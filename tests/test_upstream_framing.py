"""Upstream framing (context option `upstream_framing`, the framing of the upstream-compatible mode, DESIGN §3.10) on
every STFT-family path: the register kernels (n_fft 256 / 512 / 1024, ssq and stft mode), the shared-memory kernel,
the rows path (two-pass powers of two, Bluestein lengths, > 4096), the istft kernels, batches, streams and the feeder,
against the float64 oracle framed as upstream frames (`framing="upstream"`: left pad n_fft // 2, np.pad).

The upstream-framed oracle is pinned to upstream ssqueezepy's own outputs (tests/golden/upstream_compat.npz) by the
CPU test below.  None of those goldens needs more than one reflection, so for signals of N <= n_fft // 2 samples
(where np.pad reflects again and again) "upstream = np.pad" rests on upstream's code (utils/common.py padsignal calls
np.pad), not on a golden vector."""
import os

import numpy as np
import pytest

from oracle import ssq_oracle as O

G = os.path.join(os.path.dirname(__file__), "golden")
RTOL = 1e-4


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _golden_cases():
    z = np.load(os.path.join(G, "upstream_compat.npz"))
    for ci, (N, n_fft, hop, mod, wk, fs) in enumerate(z["cases"]):
        p = f"k{ci}_"
        d = {k[len(p):]: z[k] for k in z.files if k.startswith(p)}
        yield dict(d, N=int(N), n_fft=int(n_fft), hop=int(hop), mod=bool(mod), fs=float(fs))


# ---------------------------------------------------------------------------
# CPU: the oracle
# ---------------------------------------------------------------------------
def test_upstream_framed_oracle_reproduces_upstream_outputs():
    """Sx, dSx, Tx and istft of all seven golden cases to 1e-12, and w where finite and |Sx| > 1e-3 of its maximum.
    The modulation as compat passes it: the derivative window is scaled by fs only when modulated."""
    n = 0
    for c in _golden_cases():
        n_fft, hop, w = c["n_fft"], c["hop"], c["window_fit"]
        fs = c["fs"] if c["mod"] else 1.0
        Tx, sf, ao = O.ssq_stft(c["x"], w, n_fft=n_fft, hop_len=hop, fs=fs, modulated=c["mod"], return_aux=True,
                                framing="upstream")
        assert Tx.shape == c["Tx"].shape
        assert rel(ao["Sx"], c["Sx"]) < 1e-12, (n, rel(ao["Sx"], c["Sx"]))
        assert rel(ao["dSx"], c["dSx"]) < 1e-12, (n, rel(ao["dSx"], c["dSx"]))
        assert rel(Tx, c["Tx"]) < 1e-12, (n, rel(Tx, c["Tx"]))
        strong = np.abs(c["Sx"]) > 1e-3 * np.abs(c["Sx"]).max()
        fin = strong & np.isfinite(c["w"]) & np.isfinite(ao["w"])
        assert fin.sum() > 0.1 * strong.sum()
        assert np.abs(ao["w"][fin] - np.abs(c["w"][fin])).max() < 1e-12 * sf[-1], n
        Sx = c["Sx"]
        if c["mod"]:  # undo the rotation of the frames, as compat.istft does
            Sx = Sx * np.exp(-2j * np.pi * np.arange(Sx.shape[0]) * (n_fft // 2) / n_fft)[:, None]
        xr = O.istft(Sx, w, n_fft=n_fft, hop_len=hop, N=c["N"], framing="upstream")
        assert np.abs(xr - c["istft"]).max() < 1e-12 * max(1.0, np.abs(c["istft"]).max()), n
        n += 1
    assert n == 7


def test_upstream_and_crate_framing_coincide_for_odd_n_fft():
    """For odd n_fft both framings pad (n_fft - 1) / 2 on each side; with N > n_fft // 2 one reflection reaches every
    padded sample, so the two oracles give identical arrays (shorter signals differ: see the short-signal test)."""
    rng = np.random.default_rng(3)
    for n_fft, hop, N in [(121, 3, 400), (255, 64, 1000), (1001, 250, 3000), (33, 1, 17)]:
        x = rng.standard_normal(N)
        win = np.hanning(n_fft + 2)[1:-1].copy()
        for padtype in ("reflect", "zero"):
            a = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=10.0, padtype=padtype, return_aux=True)
            b = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=10.0, padtype=padtype, return_aux=True,
                           framing="upstream")
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
            for k in a[2]:
                assert np.array_equal(a[2][k], b[2][k]), k
            Sa, _ = O.stft(x, n_fft, hop, win, padtype)
            Sb, _ = O.stft(x, n_fft, hop, win, padtype, framing="upstream")
            assert np.array_equal(Sa, Sb)
        assert np.array_equal(O.istft(Sa, win, n_fft=n_fft, hop_len=hop, N=N),
                              O.istft(Sa, win, n_fft=n_fft, hop_len=hop, N=N, framing="upstream"))
    with pytest.raises(ValueError):
        O.stft(x, 33, 1, np.hanning(33), "reflect", framing="numpy")


def test_upstream_framing_pads_short_signals_like_np_pad():
    """The oracle's upstream reflect on signals shorter than the pad: np.pad reflects with period 2 (N - 1), N = 1 is
    a constant, where the crate's framing leaves zeros."""
    x = np.array([1.0, 2.0, 3.0])
    fr = O._frames(O._pad_stft(x, 10, "reflect", "upstream"), 10, 1)
    assert np.array_equal(fr[0], [2, 1, 2, 3, 2, 1, 2, 3, 2, 1])
    assert np.array_equal(O._pad_stft(np.array([5.0]), 8, "reflect", "upstream"), np.full(8, 5.0))
    assert np.array_equal(O._pad_stft(x, 10, "zero", "upstream"), np.pad(x, [5, 4]))
    assert O._pad_stft(x, 10, "reflect")[0] == 0.0  # the crate: beyond one reflection stays zero


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
@pytest.fixture
def upstream():
    """upstream_framing on the default context (the one the `_rs` drop-in uses), reset afterwards."""
    from ssqueeze_rs_b200 import _lib
    ctx = _lib.default_context()
    ctx.set_option("upstream_framing", 1)
    try:
        yield ctx
    finally:
        ctx.set_option("upstream_framing", 0)


@pytest.fixture
def up_engine():
    """An Engine whose context frames as upstream does, reset afterwards."""
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    eng.ctx.set_option("upstream_framing", 1)
    try:
        yield eng
    finally:
        eng.ctx.set_option("upstream_framing", 0)


def _check_up(x, win, n_fft, hop, fs, expect, **kw):
    """check_ssq (every bin classified) against the upstream-framed oracle; `expect` must be in the kernel's name
    ("=name" for an exact match)."""
    from test_parity_stft import check_ssq
    from ssqueeze_rs_b200 import _lib
    oo = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=fs, return_aux=True, framing="upstream", **kw)
    rep = check_ssq(x, win, n_fft, hop, fs, oracle_out=oo, **kw)
    _assert_kernel(_lib.default_context().last_kernel_name(), expect)
    return rep


def _assert_kernel(name, expect):
    assert (name == expect[1:]) if expect.startswith("=") else (expect in name), (name, expect)


# n_fft, kernel, hops, N: edge tiles at both ends, >= 2 interior tiles, a ragged last tile; the last N of each
# register size is shorter than n_fft
SSQ_MATRIX = [
    (256, "ssq_stft256_kernel", [(64, 9001), (17, 5003), (1, 1500), (300, 30011), (64, 200)]),
    (512, "h32r", [(32, 20011), (17, 6007), (64, 12001), (1, 1300), (32, 300)]),
    (1024, "ssq_stft1024_kernel", [(256, 40009), (100, 9001), (1, 1700), (256, 700)]),
    (64, "=stft_generic_kernel", [(8, 777), (1, 300), (64, 50)]),
    (128, "=stft_generic_kernel", [(16, 2003), (3, 401)]),
    (2048, "rows", [(512, 9001)]),
    (4096, "rows", [(1024, 20011)]),
    (500, "rows", [(125, 6001)]),
    (1000, "rows", [(100, 5003)]),
    (8192, "rows", [(2048, 40009)]),
]
SSQ_CASES = [(n_fft, k, hop, N) for n_fft, k, hn in SSQ_MATRIX for hop, N in hn]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,kernel,hop,N", SSQ_CASES)
def test_upstream_ssq_stft_every_bin(upstream, n_fft, kernel, hop, N):
    """ssq_stft with upstream framing, every reassignment bin classified against the upstream-framed oracle
    (unexplained == 0, the device's w inside the fp32 bound, Tx re-accumulated over the device's bins); the options
    (zero padding, lebesgue, a gamma that gates, modulated) on the first shape of each family; then stft mode (the
    frame-pair path of the register kernels) against O.stft(framing="upstream")."""
    from ssqueeze_rs_b200 import _lib, _rs
    rng = np.random.default_rng(n_fft * 7 + hop + N)
    x = rng.standard_normal(N) * 30.0
    win = np.hanning(n_fft + 2)[1:-1].copy()
    fs = 1000.0
    _check_up(x, win, n_fft, hop, fs, kernel)
    first = (hop, N) == next((h, n) for nf, _, hn in SSQ_MATRIX if nf == n_fft for h, n in hn)
    if first:
        for kw in (dict(padtype="zero"), dict(squeezing="lebesgue"), dict(gamma=40.0), dict(modulated=True)):
            _check_up(x, win, n_fft, hop, fs, kernel, **kw)
    for padtype in ("reflect", "zero"):
        Sx, _ = _rs.stft(x, n_fft, hop, win, padtype)
        _assert_kernel(_lib.default_context().last_kernel_name(), kernel)
        So, _ = O.stft(x, n_fft, hop, win, padtype, framing="upstream")
        assert rel(Sx, So) < RTOL, (padtype, rel(Sx, So))


@pytest.mark.gpu
def test_upstream_batched_c2_geometry(up_engine):
    """Benchmark geometry (4 x 1.8 M samples, n_fft 512, hop 32) through the batched device API with upstream framing:
    every bin of frame slices at the start, the middle and the end of each channel classified against the
    upstream-framed oracle."""
    import torch
    import bench
    from test_parity_stft import check_ssq_device
    ch, n = 4, 1_800_000
    x = bench.make_neural(torch, ch, n, 30000.0, torch.device("cuda", 0), 0x5351)
    nfr = (n - 1) // 32 + 1
    slices = [(c, f0, 96) for c in range(ch) for f0 in (0, 20_000 + 777 * c, nfr - 96)]
    rep = check_ssq_device(up_engine, x, np.hanning(512), 512, 32, 30000.0, frame_slices=slices, expect_kernel="h32r",
                           framing="upstream")
    assert rep["unexplained"] == 0 and rep["bins_total"] == 257 * 96 * len(slices), rep


SHIFT_CASES = [(256, 64, 200_000, "ssq_stft256_kernel"), (512, 32, 1_800_000, "h32r"),
               (1024, 256, 400_000, "ssq_stft1024_kernel"), (128, 8, 100_000, "=stft_generic_kernel")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,n,kernel", SHIFT_CASES)
def test_upstream_framing_is_the_crate_framing_shifted_by_one_sample(n_fft, hop, n, kernel):
    """For even n_fft upstream frame f of x[:, 1:] reads the same samples as crate frame f of x (upstream pads one
    sample more on the left), and it sits in the same slot of the same tile.  So on every column where neither frame
    touches padding, Tx and Sx (stft mode, frame pairs) are bit-equal: a difference would mean that the framing
    leaks into the arithmetic of a frame.  stft mode puts two frames through one FFT (z = x_A w + i x_B w): a frame's
    fp32 result then also depends on its partner, up to four frames away, so there the compared columns also keep
    eight frames away from any frame that touches the left padding (where the two framings read different samples;
    frames at the right end read the same reflected samples in both)."""
    import torch
    from ssqueeze_rs_b200.batch import Engine
    crate, up = Engine(0), Engine(0)
    up.ctx.set_option("upstream_framing", 1)
    g = torch.Generator(device="cuda")
    g.manual_seed(n_fft + hop)
    x = torch.randn((4, n), generator=g, device="cuda") * 20
    y = x[:, 1:].contiguous()
    win = np.hanning(n_fft)
    left = n_fft // 2
    f = np.arange((n - 2) // hop + 1)
    inner = (f * hop - left >= 0) & (f * hop - left + n_fft <= n - 1)
    for name, run in (("ssq", lambda e, s: e.ssq_stft(s, win, n_fft, hop, 30000.0)),
                      ("ssq modulated", lambda e, s: e.ssq_stft(s, win, n_fft, hop, 30000.0, modulated=True)),
                      ("stft", lambda e, s: e.stft(s, win, n_fft, hop))):
        sel = inner & ((f - 8) * hop - left >= 0) if name == "stft" else inner
        cols = torch.as_tensor(f[sel], device="cuda")
        assert len(cols) > 0.9 * len(f)
        a = run(crate, x)
        _assert_kernel(crate.last_kernel_name(), kernel)
        b = run(up, y)
        _assert_kernel(up.last_kernel_name(), kernel)
        torch.cuda.synchronize()
        assert torch.equal(a[:, :, cols], b[:, :, cols]), (name, float((a[:, :, cols] - b[:, :, cols]).abs().max()))
        del a, b


ISTFT_CASES = ([(n_fft, k, hop) for n_fft, k in ((256, "istft256_tile_kernel"), (512, "istft512_tile_kernel"),
                                                  (1024, "istft1024_tile_kernel"))
                for hop in (1, n_fft // 4, n_fft + 37)]
               + [(30, "=istft_ola_kernel", 7), (128, "=istft_ola_kernel", 16), (128, "=istft_ola_kernel", 1),
                  (100, "bluestein fft_pass rows + istft_ola_kernel<rows>", 25),
                  (2048, "istft_ola_kernel<rows>", 512), (3000, "bluestein fft_pass rows + istft_ola_kernel<rows>", 750)])


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,kernel,hop", ISTFT_CASES)
def test_upstream_istft(upstream, n_fft, kernel, hop):
    """istft with upstream framing (unpad at n_fft // 2) against O.istft(framing="upstream"), window exponents
    0 / 1 / 2, on a modified spectrum with non-zero imaginary DC / Nyquist parts (irfft ignores them)."""
    from ssqueeze_rs_b200 import _lib, _rs
    N = 700 if hop == 1 else 12 * n_fft + 333
    rng = np.random.default_rng(n_fft + hop)
    x = rng.standard_normal(N) * 5.0
    win = np.hanning(n_fft + 2)[1:-1].copy()
    So, _ = O.stft(x, n_fft, hop, win, "reflect", framing="upstream")
    So = So * (1 + 0.1 * rng.standard_normal(So.shape)) + 0.05j * rng.standard_normal(So.shape)
    for wexp in (0, 1, 2):
        xr = _rs.istft(So, win, n_fft=n_fft, hop_len=hop, N=N, win_exp=wexp)
        _assert_kernel(_lib.default_context().last_kernel_name(), kernel)
        xo = O.istft(So, win, n_fft=n_fft, hop_len=hop, N=N, win_exp=wexp, framing="upstream")
        assert np.abs(xr - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30), (wexp, np.abs(xr - xo).max())


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(256, 64), (512, 32), (512, 128), (1024, 256)])
def test_compat_round_trip_register_shapes(n_fft, hop):
    """compat.stft -> compat.istft (modulated, upstream's defaults) through the register kernels: MAE < 5e-6 as in
    upstream's reconstruction test, and the forward result against the upstream-framed oracle."""
    from ssqueeze_rs_b200 import compat
    x = np.random.default_rng(n_fft + hop).standard_normal(5001)
    win = np.hanning(n_fft + 2)[1:-1].copy()
    Sx = compat.stft(x, window=win, n_fft=n_fft, hop_len=hop)
    _, _, ao = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, modulated=True, return_aux=True, framing="upstream")
    assert rel(Sx, ao["Sx"]) < RTOL
    name = compat._context().last_kernel_name()
    assert str(n_fft) in name and "generic" not in name, name
    xr = compat.istft(Sx, window=win, n_fft=n_fft, hop_len=hop, N=len(x))
    assert compat._context().last_kernel_name().startswith(f"istft{n_fft}_tile"), compat._context().last_kernel_name()
    assert np.abs(xr - x).mean() < 5e-6


def _stream_run(eng, rec, chunks, n_fft, hop, fs=30000.0, **kw):
    """Pushes rec [samples, channels] through an SsqStftStream of `eng` in the given chunk sizes; returns the frames
    concatenated and the whole-signal transform of the same engine."""
    import torch
    from ssqueeze_rs_b200.batch import SsqStftStream
    win = np.hanning(n_fft)
    xd = torch.from_numpy(rec.T.copy()).cuda()
    transform = kw.pop("transform", "ssq_stft")
    whole = eng.stft(xd, win, n_fft, hop) if transform == "stft" else eng.ssq_stft(xd, win, n_fft, hop, fs, **kw)
    st = SsqStftStream(eng, rec.shape[1], rec.shape[0], max(chunks), win, n_fft, hop, fs, transform=transform, **kw)
    assert st.total_frames == whole.shape[2]
    parts, pos, ci = [], 0, 0
    while pos < rec.shape[0]:
        c = min(chunks[ci % len(chunks)], rec.shape[0] - pos)
        parts.append(st.push(torch.from_numpy(rec[pos:pos + c].copy()).cuda()))
        pos += c
        ci += 1
    torch.cuda.synchronize()
    st.close()
    return torch.cat(parts, dim=2), whole


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,n,chunks,kernel", [
    (128, 5, 4001, [1111, 7], "=stft_generic_kernel"), (256, 64, 9001, [2500, 777], "ssq_stft256_kernel"),
    (512, 32, 20001, [7001, 333, 1], "h32r"), (1024, 256, 20001, [4100, 999], "ssq_stft1024_kernel"),
    (512, 1000, 30001, [300], "h32r"), (256, 256 + 17, 9001, [100], "ssq_stft256_kernel"),
    (512, 32, 300, [100], "h32r"), (1024, 64, 700, [64, 5], "ssq_stft1024_kernel"),
    (512, 32, 20001, [256, 4999], "h32r"), (256, 64, 9001, [128, 1000], "ssq_stft256_kernel")])
def test_upstream_stream_equals_whole_signal(up_engine, n_fft, hop, n, chunks, kernel):
    """Streams with upstream framing (the carry-over arithmetic uses the left pad): ragged chunks, hop > n_fft with
    chunks shorter than the hop, recordings shorter than n_fft, a first push of exactly n_fft // 2 samples (the first
    frame's left reflection reads x[n_fft // 2], one sample past its own last one).  ssq equals the whole-signal transform bit for bit;
    the whole-signal result of one channel is checked against the upstream-framed oracle, so the two cannot be wrong
    the same way."""
    import torch
    rng = np.random.default_rng(n_fft + hop + n)
    rec = (rng.standard_normal((n, 3)) * 20).astype(np.float32)
    got, whole = _stream_run(up_engine, rec, chunks, n_fft, hop)
    _assert_kernel(up_engine.last_kernel_name(), kernel)
    assert got.shape == whole.shape and torch.equal(got, whole), float((got - whole).abs().max())
    To, _ = O.ssq_stft(rec[:, 1].astype(np.float64), np.hanning(n_fft), n_fft=n_fft, hop_len=hop, fs=30000.0,
                       framing="upstream")
    Tw = whole[1].cpu().numpy().astype(np.complex128)
    sc = np.abs(To).max()
    assert np.abs(Tw.sum(0) - To.sum(0)).max() < 20 * RTOL * sc  # column sums do not depend on bin flips
    assert (np.abs(Tw - To) > RTOL * sc).mean() < 4e-3
    # stft mode: frame pairs of the register kernels depend on where a push starts, so fp32 rounding, not bits
    got, whole = _stream_run(up_engine, rec, chunks, n_fft, hop, transform="stft")
    err = float((got - whole).abs().max() / whole.abs().max())
    assert err < 2e-6, err
    So, _ = O.stft(rec[:, 2].astype(np.float64), n_fft, hop, np.hanning(n_fft), "reflect", framing="upstream")
    assert rel(whole[2].cpu().numpy().astype(np.complex128), So) < RTOL


@pytest.mark.gpu
def test_upstream_recording_feeder(up_engine):
    """The host feeder behind an upstream-framed stream equals the whole-signal transform bit for bit (ssq, modulated
    ssq) and to fp32 rounding in stft mode."""
    import torch
    from ssqueeze_rs_b200.batch import RecordingFeeder
    rng = np.random.default_rng(8)
    rec = (rng.standard_normal((30_001, 3)) * 20).astype(np.float32)
    xd = torch.from_numpy(rec.T.copy()).cuda()
    for n_fft, hop in ((512, 32), (1024, 256), (256, 64)):
        win = np.hanning(n_fft)
        for mod in (False, True):
            whole = up_engine.ssq_stft(xd, win, n_fft, hop, 30000.0, modulated=mod)
            with RecordingFeeder(up_engine, rec, win, n_fft, hop, 30000.0, chunk=7777, modulated=mod) as feed:
                got = torch.cat([t.clone() for t in feed], dim=2)
            torch.cuda.synchronize()
            assert torch.equal(got, whole), (n_fft, hop, mod)
        whole = up_engine.stft(xd, win, n_fft, hop)
        with RecordingFeeder(up_engine, rec, win, n_fft, hop, chunk=7777, transform="stft") as feed:
            got = torch.cat([t.clone() for t in feed], dim=2)
        assert float((got - whole).abs().max() / whole.abs().max()) < 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,N", [(121, 3, 400), (255, 7, 1000), (1001, 100, 5000), (121, 1, 61)])
def test_upstream_odd_n_fft_is_the_crate_framing(upstream, n_fft, hop, N):
    """Odd n_fft: both framings pad (n_fft - 1) / 2 on each side, and with N > n_fft // 2 one reflection reaches
    every padded sample: the upstream-framed context computes the crate's ssq_stft, stft and istft bit for bit."""
    from ssqueeze_rs_b200 import _rs
    x = np.random.default_rng(n_fft + N).standard_normal(N)
    win = np.hanning(n_fft + 2)[1:-1].copy()
    out = {}
    for opt in (1, 0):
        upstream.set_option("upstream_framing", opt)
        Tx, _, aux = _rs.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=100.0, return_aux=True)
        Sx, _ = _rs.stft(x, n_fft, hop, win, "reflect")
        xr = _rs.istft(Sx, win, n_fft=n_fft, hop_len=hop, N=N)
        out[opt] = (Tx, aux["Sx"], aux["w"], aux["kb"], Sx, xr)
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


SHORT_NFFT = [(256, "ssq_stft256_kernel"), (512, "h32r"), (1024, "ssq_stft1024_kernel"), (2048, "rows"),
              (1000, "rows")]
SHORT_CASES = [(n_fft, k, N) for n_fft, k in SHORT_NFFT
               for N in sorted({1, 2, 3, n_fft // 4, n_fft // 2, n_fft // 2 + 1})]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,kernel,N", SHORT_CASES)
def test_upstream_reflect_of_short_signals(upstream, n_fft, kernel, N):
    """Signals of N <= n_fft // 2 samples, where upstream's np.pad reflects more than once (a 1-sample signal becomes
    a constant) and the crate's rule leaves zeros; n_fft // 2 + 1 is the first length where the two agree.  Through
    `_rs` with the option set, through compat, and through a stream, against the upstream-framed oracle.  The register
    sizes hand N <= n_fft // 2 to the shared-memory kernel, which folds.  (np.pad is what upstream's padsignal calls;
    no golden vector of upstream covers this regime.)"""
    import torch
    from ssqueeze_rs_b200 import _lib, _rs, compat
    from ssqueeze_rs_b200.batch import Engine
    if N <= n_fft // 2 and kernel != "rows":
        kernel = "=stft_generic_kernel"
    rng = np.random.default_rng(n_fft + N)
    x = rng.standard_normal(N) * 3.0 + 1.0
    win = np.hanning(n_fft)
    hop = max(1, n_fft // 8)
    # _rs (the default context, option set): stft and ssq_stft
    Sx, _ = _rs.stft(x, n_fft, hop, win, "reflect")
    name = _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, n_fft, hop, win, "reflect", framing="upstream")
    assert rel(Sx, So) < RTOL, rel(Sx, So)
    _assert_kernel(name, kernel)
    Tx, _, aux = _rs.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=1000.0, return_aux=True)
    _assert_kernel(_lib.default_context().last_kernel_name(), kernel)
    To, _, ao = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, fs=1000.0, return_aux=True, framing="upstream")
    assert rel(aux["Sx"], ao["Sx"]) < RTOL and rel(aux["dSx"], ao["dSx"]) < 2 * RTOL
    assert np.abs(Tx.sum(0) - To.sum(0)).max() < 1e-3 * np.abs(To).max()
    # compat (its own upstream-framed context; modulated, upstream's default)
    Tc, Sc, *_ = compat.ssq_stft(x, window=win, n_fft=n_fft, hop_len=hop)
    _assert_kernel(compat._context().last_kernel_name(), kernel)
    Tm, _, am = O.ssq_stft(x, win, n_fft=n_fft, hop_len=hop, modulated=True, return_aux=True, framing="upstream")
    assert rel(Sc, am["Sx"]) < RTOL, rel(Sc, am["Sx"])
    assert np.abs(Tc.sum(0) - Tm.sum(0)).max() < 1e-3 * np.abs(Tm).max()
    # a stream (two channels) in chunks of N // 2: with N <= n_fft // 2 every frame covers the whole recording and is
    # computed after the last push; with N = n_fft // 2 + 1 the first frame's left reflection reads x[n_fft // 2], one
    # sample past the frame's own last one, so it must wait for that sample
    eng = Engine(0)
    eng.ctx.set_option("upstream_framing", 1)
    rec = np.stack([x, -x], axis=1).astype(np.float32)
    got, whole = _stream_run(eng, rec, [max(1, N // 2)], n_fft, hop, fs=1000.0)
    _assert_kernel(eng.last_kernel_name(), kernel)
    To32, _ = O.ssq_stft(rec[:, 0].astype(np.float64), win, n_fft=n_fft, hop_len=hop, fs=1000.0, framing="upstream")
    Tw = whole[0].cpu().numpy().astype(np.complex128)
    assert np.abs(Tw.sum(0) - To32.sum(0)).max() < 1e-3 * np.abs(To32).max()
    assert torch.equal(got, whole), float((got - whole).abs().max())

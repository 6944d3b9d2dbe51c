"""Streaming inverse (ssq_istream_*, `IstftStream`, DESIGN §3.4c): istft and issq_stft over chunks of frames equal the
batch call on the whole Sx / Tx -- bit for bit in one push, and in pushes that keep the tile kernels' tiles where the
batch call puts them; to fp32 rounding in ragged pushes -- on every kernel family.  Argument checks run without a GPU."""
import ctypes as C

import numpy as np
import pytest

RAGGED = [1, 7, 333, 4096, 1000]

# (n_fft, hop, the kernel the overlap-add must reach)
FAMILIES = [(512, 32, "istft512_tile_kernel"), (512, 100, "istft512_tile_kernel"),
            (256, 64, "istft256_tile_kernel"), (1024, 256, "istft1024_tile_kernel"),
            (128, 5, "istft_ola_kernel"), (2048, 512, "fft_pass rows + istft_ola_kernel<rows>"),
            (500, 125, "bluestein fft_pass rows + istft_ola_kernel<rows>")]


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU: the ABI checks its arguments before it looks at the context
# ---------------------------------------------------------------------------------------------------------------------
def _create(lib, ctx=None, channels=2, n_frames=100, n_out=0, max_frames=10, n_fft=512, hop=32, win_exp=1, mode=0,
            fs=1.0, out_format=0):
    w = np.hanning(n_fft)
    h = C.c_void_p()
    st = lib.ssq_istream_create(ctx, channels, n_frames, n_out, max_frames, C.c_void_p(w.ctypes.data), len(w), n_fft,
                                hop, win_exp, mode, fs, out_format, C.byref(h))
    return st, (lib.ssq_last_error(None) or b"").decode()


def test_istream_argument_validation_without_gpu(built_lib):
    from ssqueeze_rs_b200._lib import SSQ_EINVAL
    lib = built_lib
    st, msg = _create(lib, mode=2)
    assert st == SSQ_EINVAL and "mode" in msg
    st, msg = _create(lib, out_format=3)
    assert st == SSQ_EINVAL and "out_format" in msg
    st, msg = _create(lib, out_format=-1)
    assert st == SSQ_EINVAL and "out_format" in msg
    st, msg = _create(lib, mode=1, hop=2)
    assert st == SSQ_EINVAL and "hop_len != 1" in msg
    st, msg = _create(lib, mode=1, hop=1, n_out=99)
    assert st == SSQ_EINVAL and "one sample per frame" in msg
    for bad in (dict(max_frames=0), dict(channels=0), dict(n_frames=0), dict(n_fft=1), dict(hop=0), dict(win_exp=-1)):
        st, msg = _create(lib, **bad)
        assert st == SSQ_EINVAL and "bad sizes" in msg, bad
    st, msg = _create(lib)  # valid arguments: only then the missing context
    assert st == SSQ_EINVAL and "ctx is NULL" in msg
    n = C.c_int64(7)
    assert lib.ssq_istream_push(None, None, 1, 1.0, None, C.byref(n)) == SSQ_EINVAL
    assert lib.ssq_istream_samples_after(None, 5) == 0 and lib.ssq_istream_total_samples(None) == 0
    lib.ssq_istream_destroy(None)


def test_istft_stream_python_argument_errors_without_gpu(built_lib):
    from ssqueeze_rs_b200.batch import IstftStream
    with pytest.raises(ValueError, match="transform"):
        IstftStream(None, 2, 100, 10, np.hanning(512), transform="icwt")
    with pytest.raises(ValueError, match="out must be"):
        IstftStream(None, 2, 100, 10, np.hanning(512), out="i32")


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
def _signal(channels, n, seed):
    import torch
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 30000.0
    x = (rng.standard_normal((channels, n)) * 20 + 50 * np.sin(2 * np.pi * 700 * t)).astype(np.float32)
    return torch.from_numpy(x).cuda()


def _push_all(eng, Sx, win, n_fft, hop, schedule, N=None, win_exp=1, out="f32", scale=1.0, transform="istft",
              fs=1.0, kernels=None, between=None):
    """Pushes Sx [channels, n_freqs, n_frames] in chunks cycling through `schedule`; returns the output in the
    [channels, samples] layout (int16 or float32 as `out` says)."""
    import torch
    from ssqueeze_rs_b200.batch import IstftStream
    ch, nfq, nfr = Sx.shape
    inv = IstftStream(eng, ch, nfr, max(schedule), win, n_fft, hop, N=N, win_exp=win_exp, transform=transform, fs=fs,
                      out=out, scale=scale)
    parts, pos, i = [], 0, 0
    while pos < nfr:
        k = min(schedule[i % len(schedule)], nfr - pos)
        y = inv.push(Sx[:, :, pos:pos + k].contiguous())
        if kernels is not None:
            kernels.add(eng.last_kernel_name())
        parts.append(y.clone() if out == "f32" else y.t().clone())
        pos += k
        i += 1
        if between is not None:
            between()
    torch.cuda.synchronize()
    got = torch.cat(parts, dim=1)
    assert got.shape[1] == inv.total_samples
    inv.close()
    return got


def _case(n_fft, hop, channels=3, frames=6000, N=None, seed=0):
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    n = hop * frames
    x = _signal(channels, n, seed + n_fft + hop)
    win = np.hanning(n_fft)
    Sx = eng.stft(x, win, n_fft, hop)
    return eng, win, Sx


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,kernel", FAMILIES)
def test_one_push_equals_the_batch_call_bit_for_bit(n_fft, hop, kernel):
    eng, win, Sx = _case(n_fft, hop, frames=3000)
    whole = eng.istft(Sx, win, n_fft, hop)
    assert eng.last_kernel_name() == kernel
    seen = set()
    got = _push_all(eng, Sx, win, n_fft, hop, [Sx.shape[2]], kernels=seen)
    assert seen == {kernel}
    assert got.shape == whole.shape
    assert bool((got == whole).all()), float((got - whole).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,tile,kernel", [(512, 32, 32, "istft512_tile_kernel"),
                                                  (256, 64, 32, "istft256_tile_kernel"),
                                                  (1024, 256, 8, "istft1024_tile_kernel")])
def test_pushes_in_multiples_of_the_tile_are_bit_equal(n_fft, hop, tile, kernel):
    """Tiles of the stream start where the batch call's start, and no sample is covered by more than two tiles: each
    sample is the same one- or two-term sum, carried across a seam or added by two atomics."""
    eng, win, Sx = _case(n_fft, hop, frames=2011)
    whole = eng.istft(Sx, win, n_fft, hop)
    seen = set()
    got = _push_all(eng, Sx, win, n_fft, hop, [tile, 3 * tile, 10 * tile, 2 * tile], kernels=seen)
    assert seen == {kernel}
    assert bool((got == whole).all()), float((got - whole).abs().max())


def _close(got, whole, tol=2e-6):
    err = float((got - whole).abs().max() / whole.abs().max())
    assert err <= tol, err


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,kernel", FAMILIES)
def test_ragged_pushes_in_every_family(n_fft, hop, kernel):
    eng, win, Sx = _case(n_fft, hop, frames=9000 if hop < 100 else 5200)
    whole = eng.istft(Sx, win, n_fft, hop)
    seen = set()
    got = _push_all(eng, Sx, win, n_fft, hop, RAGGED, kernels=seen)
    assert seen == {kernel}
    assert got.shape == whole.shape
    _close(got, whole)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 600), (128, 200), (1024, 256)])
@pytest.mark.parametrize("n_mode", ["short", "long"])
def test_ragged_pushes_hop_beyond_n_fft_and_other_lengths(n_fft, hop, n_mode):
    """hop > n_fft (gaps no frame covers come out 0); N < hop * n_frames drops the frames past max_hops, N > hop *
    n_frames appends a zero tail.  With hop >= n_fft every sample is one frame's w * x divided by w^2, which is tiny at
    the ends of a Hann window: the fp32 rounding of that frame is amplified there.  The n_fft 512 kernel transforms
    frames in pairs (2k, 2k + 1) of its push, so there the pushes have even sizes: every frame keeps the batch call's
    partner and the result is bit-equal; the generic kernel (128) transforms frames one by one and takes odd sizes."""
    eng, win, Sx = _case(n_fft, hop, frames=1500)
    nfr = Sx.shape[2]
    N = hop * nfr - 7 * hop - 3 if n_mode == "short" else hop * nfr + 5 * hop + 11
    whole = eng.istft(Sx, win, n_fft, hop, N=N)
    if n_fft == 512:
        got = _push_all(eng, Sx, win, n_fft, hop, [2, 8, 334, 100, 2], N=N)
        assert bool((got == whole).all()), float((got - whole).abs().max())
    else:
        got = _push_all(eng, Sx, win, n_fft, hop, [1, 7, 333, 100, 2], N=N)
        _close(got, whole)
    assert got.shape == whole.shape == (3, N)
    one = _push_all(eng, Sx, win, n_fft, hop, [nfr], N=N)
    assert bool((one == whole).all())


@pytest.mark.gpu
@pytest.mark.parametrize("win_exp", [0, 2])
@pytest.mark.parametrize("n_fft,hop", [(512, 32), (128, 5)])
def test_ragged_pushes_other_window_exponents(win_exp, n_fft, hop):
    eng, win, Sx = _case(n_fft, hop, frames=5000)
    whole = eng.istft(Sx, win, n_fft, hop, win_exp=win_exp)
    got = _push_all(eng, Sx, win, n_fft, hop, RAGGED, win_exp=win_exp)
    _close(got, whole)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 32), (511, 32), (256, 64), (255, 64)])
def test_ragged_pushes_upstream_framing(n_fft, hop):
    """With upstream_framing the stream unpads at n_fft // 2, as the batch call does: even and odd n_fft differ."""
    from oracle import ssq_oracle as O
    eng, win, Sx = _case(n_fft, hop, frames=4000)
    eng.ctx.set_option("upstream_framing", 1)
    whole = eng.istft(Sx, win, n_fft, hop)
    got = _push_all(eng, Sx, win, n_fft, hop, RAGGED)
    _close(got, whole)
    one = _push_all(eng, Sx, win, n_fft, hop, [Sx.shape[2]])
    assert bool((one == whole).all())
    ref = O.istft(Sx[0].cpu().numpy().astype(np.complex128), win, n_fft=n_fft, hop_len=hop, framing="upstream")
    err = np.abs(got[0].cpu().numpy() - ref).max() / np.abs(ref).max()
    assert err <= 1e-4, err
    eng.ctx.set_option("upstream_framing", 0)
    crate = eng.istft(Sx, win, n_fft, hop)
    if n_fft % 2 == 0:
        assert not bool((crate == whole).all())  # one sample apart
    else:
        assert bool((crate == whole).all())


@pytest.mark.gpu
def test_ragged_schedule_is_deterministic_and_ignores_batch_calls_in_between():
    import torch
    eng, win, Sx = _case(512, 32, frames=6000)
    a = _push_all(eng, Sx, win, 512, 32, RAGGED)
    b = _push_all(eng, Sx, win, 512, 32, RAGGED)
    assert bool((a == b).all())
    other = eng.stft(_signal(2, 40000, 9), np.kaiser(256, 8.0), 256, 17)

    def batch_call():  # another window, n_fft, hop and size: replaces the context's tables and workspace
        eng.istft(other, np.kaiser(256, 8.0), 256, 17, win_exp=2)
    c = _push_all(eng, Sx, win, 512, 32, RAGGED, between=batch_call)
    torch.cuda.synchronize()
    assert bool((a == c).all())


@pytest.mark.gpu
@pytest.mark.parametrize("framing", ["crate", "upstream"])
def test_stream_against_the_float64_oracle(framing):
    from oracle import ssq_oracle as O
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    if framing == "upstream":
        eng.ctx.set_option("upstream_framing", 1)
    x = _signal(1, 96000, 5)
    win = np.hanning(512)
    Sx = eng.stft(x, win, 512, 32)
    got = _push_all(eng, Sx, win, 512, 32, RAGGED, N=96000)[0].cpu().numpy()
    ref = O.istft(Sx[0].cpu().numpy().astype(np.complex128), win, n_fft=512, hop_len=32, N=96000, framing=framing)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err <= 1e-4, err


@pytest.mark.gpu
def test_samples_after_and_errors_leave_the_stream_intact():
    import torch
    from ssqueeze_rs_b200 import _lib
    from ssqueeze_rs_b200.batch import IstftStream
    eng, win, Sx = _case(512, 32, channels=2, frames=700)
    nfr = Sx.shape[2]
    whole = eng.istft(Sx, win, 512, 32)
    inv = IstftStream(eng, 2, nfr, 400, win, 512, 32)
    lib = _lib.load()
    assert inv.total_samples == 32 * nfr
    assert lib.ssq_istream_samples_after(inv._h, 1) == 0  # frame 0 ends before output 0 (left = 255) is final
    assert lib.ssq_istream_samples_after(inv._h, 10) == 10 * 32 - 255
    assert lib.ssq_istream_samples_after(inv._h, nfr) == 32 * nfr
    parts = [inv.push(Sx[:, :, :10].contiguous())]
    assert parts[0].shape == (2, 65)
    assert lib.ssq_istream_samples_after(inv._h, 5) == 5 * 32
    with pytest.raises(ValueError, match="max_frames"):
        inv.push(Sx[:, :, 10:411].contiguous())
    w = C.c_int64(-1)
    chunk = Sx[:, :, 10:20].contiguous()
    st = lib.ssq_istream_push(inv._h, C.c_void_p(chunk.data_ptr()), 10, 1.0, None, C.byref(w))
    with pytest.raises(ValueError, match="d_out is NULL"):
        _lib.raise_status(st, eng.ctx.handle)
    assert w.value == 0
    parts.append(inv.push(Sx[:, :, 10:300].contiguous()))
    parts.append(inv.push(Sx[:, :, 300:nfr - 1].contiguous()))
    with pytest.raises(ValueError, match="n_frames_total"):
        inv.push(Sx[:, :, nfr - 2:].contiguous())
    parts.append(inv.push(Sx[:, :, nfr - 1:].contiguous()))
    torch.cuda.synchronize()
    got = torch.cat(parts, dim=1)
    assert lib.ssq_istream_samples_after(inv._h, 1) == 0
    _close(got, whole)  # pushes of 10, 290, 399 and 1 frames: not multiples of the tile
    inv.close()


def _i16_rule(y, scale):
    """np.clip(np.rint(y * float32(1 / scale))) as int16, y float32"""
    return np.clip(np.rint(y * np.float32(1.0 / scale)), -32768, 32767).astype(np.int16)


@pytest.mark.gpu
def test_file_to_file_band_stop_through_the_forward_and_inverse_streams(tmp_path):
    import torch
    from ssqueeze_rs_b200.batch import Engine, IstftStream, RecordingFeeder
    eng = Engine(0)
    n, ch, chunk, scale = 150_001, 4, 7777, 0.195
    rng = np.random.default_rng(11)
    t = np.arange(n) / 30000.0
    sig = rng.standard_normal((n, ch)) * 300 + 4000 * np.sin(2 * np.pi * 1500 * t)[:, None]
    src = np.memmap(tmp_path / "in.dat", dtype=np.int16, mode="w+", shape=(n, ch))
    src[:] = np.clip(np.rint(sig), -32768, 32767).astype(np.int16)
    src.flush()
    rec = np.memmap(tmp_path / "in.dat", dtype=np.int16, mode="r").reshape(-1, ch)
    win = np.hanning(512)
    nfr = (n - 1) // 32 + 1
    max_frames = (chunk + 512) // 32 + 2
    band = torch.ones((1, 257, 1), dtype=torch.float32, device="cuda")
    band[:, 20:35] = 0.0  # 1.2 - 2.0 kHz at 30 kHz: removes the sine
    x = torch.from_numpy((np.asarray(rec).astype(np.float32) * np.float32(scale)).T.copy()).cuda()
    Sx_whole = eng.stft(x, win, 512, 32)
    for name, mask in (("stop", band), ("identity", torch.ones_like(band))):
        out = np.memmap(tmp_path / f"{name}.dat", dtype=np.int16, mode="w+", shape=(n, ch))
        pos = 0
        with IstftStream(eng, ch, nfr, max_frames, win, 512, 32, N=n, out="i16_interleaved", scale=scale) as inv, \
                RecordingFeeder(eng, rec, win, 512, 32, chunk=chunk, scale=scale, transform="stft") as feed:
            for Sx in feed:
                y = inv.push(mask * Sx)
                out[pos:pos + y.shape[0]] = y.cpu().numpy()
                pos += y.shape[0]
        assert pos == n
        out.flush()
        got = np.asarray(np.memmap(tmp_path / f"{name}.dat", dtype=np.int16, mode="r").reshape(-1, ch))
        ref = _i16_rule(eng.istft(mask * Sx_whole, win, 512, 32, N=n).cpu().numpy(), scale).T
        d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
        # the stft-mode stream pairs frames differently from the whole-signal transform (fp32 rounding, see
        # test_stream.py): an output that lies at a rounding boundary may come out one count apart
        assert d.max() <= 1, d.max()
        print(f"{name}: {int((d == 1).sum())} of {d.size} counts differ by 1")
        if name == "identity":
            assert np.abs(got.astype(np.int32) - np.asarray(rec).astype(np.int32)).max() <= 1
        else:  # the sine is gone, the noise stays
            assert got.astype(np.float64).std() < 0.5 * np.asarray(rec).astype(np.float64).std()


@pytest.mark.gpu
@pytest.mark.parametrize("out,scale", [("f32", 1.0), ("f32", 0.5), ("f32_interleaved", 1.0),
                                       ("i16_interleaved", 0.195)])
def test_issq_stft_stream_from_the_modulated_forward_stream(out, scale):
    import torch
    from ssqueeze_rs_b200.batch import Engine, IstftStream, SsqStftStream
    eng = Engine(0)
    n, ch, fs = 20_011, 3, 30000.0
    rng = np.random.default_rng(3)
    rec = (rng.standard_normal((n, ch)) * 20).astype(np.float32)
    win = np.hanning(512)
    chunks = [1, 777, 5000, 3333]
    fwd = SsqStftStream(eng, ch, n, max(chunks), win, 512, 1, fs, modulated=True)
    inv = IstftStream(eng, ch, n, max(chunks) + 512 + 2, win, 512, 1, transform="issq_stft", fs=fs, out=out,
                      scale=scale)
    Tx_parts, y_parts, pos, i = [], [], 0, 0
    while pos < n:
        k = min(chunks[i % len(chunks)], n - pos)
        Tx = fwd.push(torch.from_numpy(rec[pos:pos + k].copy()).cuda())
        Tx_parts.append(Tx)
        y_parts.append(inv.push(Tx))
        assert eng.last_kernel_name() == "istream_issq_kernel" or Tx.shape[2] == 0
        pos += k
        i += 1
    torch.cuda.synchronize()
    whole = eng.issq_stft(torch.cat(Tx_parts, dim=2), win, 512, fs).cpu().numpy()
    got = torch.cat(y_parts, dim=1 if out == "f32" else 0).cpu().numpy()
    if out != "f32":
        got = got.T
    assert got.shape == whole.shape == (ch, n)
    if out == "i16_interleaved":
        assert np.array_equal(got, _i16_rule(whole, scale))
    else:
        assert np.array_equal(got, whole * np.float32(1.0 / scale))
    fwd.close()
    inv.close()

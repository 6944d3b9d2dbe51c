"""Every kernel family at the sizes the project is run at: output tensors past 2^31 (and 2^32) elements, and work
that the host planners cut into two or more blocks.

Each GPU case uses two references:
1. Per-channel identity.  The big batch is computed once; sampled channels are recomputed alone in small calls, where
   the planners choose other blocks and offsets, and must come out bit for bit the same (channels are independent).
   Two families are not bit-equal and are held to a stated bound instead: the fused ssq_cwt tail (its bins are
   equal), and istft where a sample collects more than two tile sums (`_istft_same`).
2. The float64 oracle on the sampled channels: slices of frames at the start, at every block seam and at the end with
   every bin classified (`check_ssq_device`), `O.istft` on whole channels, and the component / inverse references
   on column slices (each column of those is a sum over rows).

Sampled channels: 0 and the last, the channels holding output element 2^31 and 2^32, and the first and last channel
of every planner block.  The planner blocks come from the restatements below, each citing the source it restates; the
tests without a GPU assert that the chosen geometries really span two or more blocks.

Out of reach: the tile-count fallback of the register kernels (total_tiles > 0x7ff00000) needs on the order of 10^14
bytes of Tx.
"""
import gc

import numpy as np
import pytest

from oracle import ridge_oracle as R
from oracle import ssq_oracle as O

RTOL = 1e-4
EPS32 = float(np.finfo(np.float32).eps)
SSQ_EUNSUPPORTED = 4
FFT_MAX_ROWS = 65535  # gridDim.y of the row passes (fft_run, cwt_host.inl)


# ---------------------------------------------------------------------------------------------------------------------
# the host planners, restated
# ---------------------------------------------------------------------------------------------------------------------
def rows_plan(n_fft, channels, n_frames):
    """stft_rows_run / istft_rows_run (stft_rows.inl): rows of M = 2^k >= n_fft points (Bluestein: >= 2 n_fft - 1),
    at most rows_max = min(65 535, 512 MiB / (8 M)) rows per launch, channel blocks of cc_max = min(channels,
    rows_max), frame blocks of fb = rows_max / cc.  -> M, rows_max, [(c0, cc, f0, nf), ...]."""
    pow2 = n_fft & (n_fft - 1) == 0
    assert not (n_fft <= 1024 if pow2 else n_fft <= 32), "shared-memory kernel, not the rows path (stft_rows_skip)"
    M = 1
    while M < (n_fft if pow2 else 2 * n_fft - 1):
        M <<= 1
    rows_max = max(2, min(FFT_MAX_ROWS, (512 << 20) // (8 * M)))
    cc_max = min(channels, rows_max)
    blocks = []
    for c0 in range(0, channels, cc_max):
        cc = min(cc_max, channels - c0)
        fb = max(1, rows_max // cc)
        for f0 in range(0, n_frames, fb):
            blocks.append((c0, cc, f0, min(fb, n_frames - f0)))
    return M, rows_max, blocks


def ridge_plan(F, Tn, channels, itemsize):
    """ridge_run (ridge_host.inl): time tile TT = 32 halved until the backward pass's two [F][TT + 1] tiles (plus a
    row and 64 ints) fit 200 KiB of shared memory (None: not even at TT = 1); channel batches cb of 20 GiB of three
    [F, Tn] maps.  -> (TT, cb)."""
    def smem(tt):
        return (2 * F * (tt + 1) + F) * itemsize + 64 * 4
    TT = 32
    while TT > 1 and smem(TT) > 200 * 1024:
        TT >>= 1
    if smem(TT) > 200 * 1024:
        return None
    return TT, max(1, min(channels, (20 << 30) // (F * Tn * itemsize)))


def ridge_rows_limit(itemsize):
    """The most rows ridge_run takes in this real type: 8192, or fewer where two tiles do not fit at TT = 1."""
    return min(8192, (200 * 1024 - 64 * 4) // (5 * itemsize))


def n_frames(n, hop):
    return (n - 1) // hop + 1


# geometries of the GPU cases below
ROWS_REGRESSION = [  # (channels, n, n_fft, hop): one launch of more than 65 535 rows before the cap
    (16, 30_000, 255, 7),
    (100, 30_000, 100, 10),
]
ROWS_SEAMS = [  # (channels, n, n_fft, hop): frame blocks (2048) and channel blocks (8192, Bluestein 3000)
    (2, 1_200_000, 2048, 32),
    (8200, 10_000, 8192, 2500),
    (8200, 6_001, 3000, 1500),
]
RIDGE_ROWS_F32 = [(763, 32), (764, 16), (1025, 16), (2047, 8), (4096, 4), (8192, 1)]  # (F, TT)
RIDGE_BATCH = (373, 257, 56_250)  # channels, F, Tn: cb = 371 -> two batches


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU: the geometries reach what they are meant to reach
# ---------------------------------------------------------------------------------------------------------------------
def test_rows_planner_caps_every_launch_and_the_cases_cross_seams():
    # the regression cases: the uncapped planner (512 MiB / (8 M) rows) put more than 65 535 rows into one launch
    for ch, n, nf_, hop in ROWS_REGRESSION + [(1, 70_000, 300, 1)]:
        M, rows_max, blocks = rows_plan(nf_, ch, n_frames(n, hop))
        uncapped = max(2, (512 << 20) // (8 * M))
        first = min(ch, uncapped) * min(max(1, uncapped // min(ch, uncapped)), n_frames(n, hop))
        assert first > FFT_MAX_ROWS, (ch, n, nf_, hop, first)
        assert all(cc * nf <= FFT_MAX_ROWS for _, cc, _, nf in blocks)
        assert len(blocks) >= 2
    # the seam cases: frame blocks (one channel block, several frame blocks) and channel blocks
    M, rows_max, blocks = rows_plan(2048, 2, n_frames(1_200_000, 32))
    assert (M, rows_max) == (2048, 32768) and len({b[0] for b in blocks}) == 1 and len(blocks) >= 3
    for ch, n, nf_, hop in ROWS_SEAMS[1:]:
        M, rows_max, blocks = rows_plan(nf_, ch, n_frames(n, hop))
        assert (M, rows_max) == (8192, 8192)
        assert len({b[0] for b in blocks}) >= 2 and len(blocks) >= 3, blocks
        assert ch > rows_max
    for ch, n, nf_, hop in ROWS_SEAMS:
        assert all(cc * nf <= FFT_MAX_ROWS for _, cc, _, nf in rows_plan(nf_, ch, n_frames(n, hop))[2])


def test_ridge_planner_tiles_batches_and_limits():
    for F, TT in RIDGE_ROWS_F32:
        assert ridge_plan(F, 37, 1, 4)[0] == TT, F
    assert ridge_plan(1025, 37, 1, 4)[0] < 32 and 1025 > 1024  # both kernels loop over f (1024 threads)
    ch, F, Tn = RIDGE_BATCH
    assert ridge_plan(F, Tn, ch, 4)[1] == 371 and ch >= 372
    # double: two tiles of 5113 rows fit at TT = 1, of 5114 do not
    assert ridge_rows_limit(8) == 5113 and ridge_rows_limit(4) == 8192
    assert ridge_plan(5113, 13, 1, 8)[0] == 1 and ridge_plan(5114, 13, 1, 8) is None
    assert ridge_plan(8192, 13, 1, 4)[0] == 1


def test_sampled_channels_hold_the_elements_past_2_31():
    per = 257 * n_frames(1_800_000, 32)
    assert _sampled(384, per) == [0, 148, 297, 383]
    assert _sampled(8, 576 << 20) == [0, 3, 7]


# ---------------------------------------------------------------------------------------------------------------------
# helpers of the GPU cases
# ---------------------------------------------------------------------------------------------------------------------
def _sampled(ch, per_ch, extra=()):
    s = {0, ch - 1, *extra}
    for e in (1 << 31, 1 << 32):
        if e < ch * per_ch:
            s.add(e // per_ch)
    return sorted(s)


def _free_and_need(nbytes):
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 1e9:.1f} GB of device memory, {free / 1e9:.1f} GB free")


def _signals(ch, n, seed, scale=3.0):
    """float32 CUDA [ch, n]: per channel its own seed and a tone at a channel-dependent frequency (cycles per sample),
    so that a swapped or shifted channel cannot match."""
    import torch
    x = torch.empty((ch, n), dtype=torch.float32, device="cuda")
    t = torch.arange(n, device="cuda", dtype=torch.float64)
    g = torch.Generator(device="cuda")
    for c in range(ch):
        g.manual_seed(seed * 1_000_003 + c)
        f = 0.01 + 0.45 * ((c * 0.6180339887) % 1.0)
        x[c] = torch.randn(n, generator=g, device="cuda") * scale + (2 * scale * torch.sin(2 * np.pi * f * t)).float()
    return x


def _stft_slices(nfr, hop, n_fft, blocks_f0=(), elems=(), span=64):
    """(first_frame, n_frames) slices at the start, at every seam frame and element frame, and at the end."""
    s = [(0, min(span, nfr)), (max(0, nfr - span), min(span, nfr))]
    s += [(max(0, f - span // 2), min(span, nfr - max(0, f - span // 2))) for f in list(blocks_f0) + list(elems)]
    return sorted(set(s))


def _check_stft_slices(Sx_c, x_c, win, n_fft, hop, slices):
    """Sx of one channel (device) against O.stft on the samples of each slice of frames (check_ssq_device's slicing:
    slice frame j is global frame g0 + j)."""
    import torch
    n = x_c.shape[0]
    left = O.pad_left(n_fft)
    for f0, nf in slices:
        g0 = max(0, (f0 * hop - left) // hop)
        a, b = g0 * hop, min(n, (f0 + nf - 1) * hop - left + n_fft)
        So, _ = O.stft(x_c[a:b].cpu().numpy().astype(np.float64), n_fft, hop, win, "reflect")
        sel = np.arange(f0 - g0, min(f0 - g0 + nf, So.shape[1]))
        got = Sx_c[:, torch.as_tensor(g0 + sel, device=Sx_c.device)].cpu().numpy().astype(np.complex128)
        ref = So[:, sel]
        assert np.abs(got - ref).max() < RTOL * np.abs(ref).max(), (f0, nf)


def _istft_vs_oracle(xr_c, Sx_c, win, n_fft, hop, n):
    xo = O.istft(Sx_c.cpu().numpy().astype(np.complex128), win, n_fft=n_fft, hop_len=hop, N=n)
    got = xr_c.cpu().numpy().astype(np.float64)
    assert np.abs(got - xo).max() < RTOL * max(np.abs(xo).max(), 1e-30)


def _istft_same(one, batch, exact, n_fft, hop):
    """A channel of the one-channel istft against the same channel of the batch.  The tile kernels sum the frames of
    a tile and merge tile seams with float atomics: bit-equal where a sample collects at most two tile sums (exact),
    else the order of the CTAs changes the last bits, bounded by the reordering of ceil(n_fft / hop) contributions of
    one sign (consistent Sx: each is x[p] w^(a+1))."""
    import torch
    if exact:
        assert torch.equal(one, batch)
        return
    lim = 2 * -(-n_fft // hop) * EPS32 * float(batch.abs().max())
    d = float((one - batch).abs().max())
    assert d <= lim, (d, lim)


# frames per tile of the istft tile kernels (istft_h32.cuh, istft_r1024.cuh, istft_r256.cuh): a sample collects at most
# two tile sums iff n_fft <= (F + 1) hop
ISTFT_TILE_FRAMES = {512: 32, 1024: 8, 256: 32}


def _engine():
    from ssqueeze_rs_b200.batch import Engine
    return Engine(0)


def _ssq_stft_family(eng, x, win, n_fft, hop, fs, sampled, slices_of, kernel):
    """ssq_stft, stft and istft of the batch x: sampled channels alone (identity) and against the oracle.
    slices_of(c): frame slices of channel c for the oracle, or None for whole channels."""
    import torch
    from test_parity_stft import check_ssq_device
    ch, n = x.shape
    Tx = eng.ssq_stft(x, win, n_fft, hop, fs)
    torch.cuda.synchronize()
    assert kernel in eng.last_kernel_name(), eng.last_kernel_name()
    for c in sampled:
        Tc = eng.ssq_stft(x[c:c + 1], win, n_fft, hop, fs)
        assert torch.equal(Tc[0], Tx[c]), c
        sl = slices_of(c)
        rep = check_ssq_device(eng, x[c:c + 1], win, n_fft, hop, fs, expect_kernel=kernel,
                               frame_slices=None if sl is None else [(0, f0, nf) for f0, nf in sl])
        assert rep["unexplained"] == 0, (c, rep)
    del Tx, Tc
    torch.cuda.empty_cache()
    Sx = eng.stft(x, win, n_fft, hop)
    torch.cuda.synchronize()
    assert kernel in eng.last_kernel_name(), eng.last_kernel_name()
    for c in sampled:
        assert torch.equal(eng.stft(x[c:c + 1], win, n_fft, hop)[0], Sx[c]), c
        sl = slices_of(c)
        _check_stft_slices(Sx[c], x[c], win, n_fft, hop, sl if sl is not None else [(0, Sx.shape[2])])
    return Sx


# ---------------------------------------------------------------------------------------------------------------------
# STFT family past 2^31 elements
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,ch,kernel", [(512, 384, "ssq_stft512_h32r_kernel"), (1024, 96, "ssq_stft1024_kernel"),
                                             (256, 320, "ssq_stft256_kernel")])
def test_ssq_stft_and_stft_past_2_31(n_fft, ch, kernel):
    """The bench geometry (1.8 M samples per channel, hop 32) with the Tx of the batch past 2^31 elements (n_fft 512:
    5.55e9, past 2^32 too): the channels holding element 2^31 / 2^32 and the ends equal the one-channel call, and
    slices of frames at the start, around those elements and at the end agree with the oracle, bin by bin."""
    import torch
    n, hop, fs = 1_800_000, 32, 30000.0
    nfq, nfr = n_fft // 2 + 1, n_frames(n, hop)
    per = nfq * nfr
    assert ch * per > 1 << 31
    _free_and_need(ch * per * 8 + ch * n * 4 + (4 << 30))
    eng = _engine()
    x = _signals(ch, n, n_fft)
    win = np.hanning(n_fft)
    sampled = _sampled(ch, per)
    elem_frames = {}
    for e in (1 << 31, 1 << 32):
        if e < ch * per:
            elem_frames.setdefault(e // per, []).append((e % per) % nfr)
    Sx = _ssq_stft_family(eng, x, win, n_fft, hop, fs, sampled,
                          lambda c: _stft_slices(nfr, hop, n_fft, elems=elem_frames.get(c, ())), kernel)
    del Sx, x, eng
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,ch,kernel", [(512, 1024, "istft512"), (1024, 480, "istft1024"), (256, 1800, "istft256")])
def test_istft_past_2_31(n_fft, ch, kernel):
    """istft of an Sx past 2^31 elements (300 k samples per channel, hop 32): sampled channels agree with O.istft on
    the whole channel and equal the one-channel call (n_fft 1024 at hop 32: to the reordering bound of _istft_same)."""
    import torch
    n, hop = 300_000, 32
    nfq, nfr = n_fft // 2 + 1, n_frames(n, hop)
    per = nfq * nfr
    assert ch * per > 1 << 31
    _free_and_need(ch * per * 8 + 2 * ch * n * 4 + (2 << 30))
    eng = _engine()
    x = _signals(ch, n, 7 + n_fft)
    win = np.hanning(n_fft)
    Sx = eng.stft(x, win, n_fft, hop)
    xr = eng.istft(Sx, win, n_fft, hop, N=n)
    torch.cuda.synchronize()
    assert kernel in eng.last_kernel_name(), eng.last_kernel_name()
    exact = n_fft <= (ISTFT_TILE_FRAMES[n_fft] + 1) * hop
    for c in _sampled(ch, per):
        _istft_vs_oracle(xr[c], Sx[c], win, n_fft, hop, n)
        _istft_same(eng.istft(Sx[c:c + 1], win, n_fft, hop, N=n)[0], xr[c], exact, n_fft, hop)
    del Sx, xr, x, eng
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# the rows path (n_fft above 1024, lengths that are not powers of two)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rows_path_one_channel_at_hop_1_past_65535_rows():
    """Upstream's default hop 1 on a Bluestein length: 70 000 frames of n_fft 300 (rows of 1024 points, 65 536 rows
    per launch before the cap) through the float64 drop-ins, forward and inverse, against the oracle."""
    from ssqueeze_rs_b200 import _lib, _rs
    from test_parity_stft import check_ssq
    rng = np.random.default_rng(300)
    n = 70_000
    x = rng.standard_normal(n) * 3.0 + 4.0 * np.sin(2 * np.pi * 0.0731 * np.arange(n))
    win = np.hanning(300)
    rep = check_ssq(x, win, 300, 1, 1.0, expect_kernel="bluestein fft_pass rows")
    assert rep["unexplained"] == 0
    Sx, _ = _rs.stft(x, 300, 1, win, "reflect")
    assert "rows" in _lib.default_context().last_kernel_name()
    So, _ = O.stft(x, 300, 1, win, "reflect")
    assert np.abs(Sx - So).max() < RTOL * np.abs(So).max()
    xr = _rs.istft(So, win, n_fft=300, hop_len=1, N=n)
    assert "istft_ola_kernel<rows>" in _lib.default_context().last_kernel_name()
    xo = O.istft(So, win, n_fft=300, hop_len=1, N=n)
    assert np.abs(xr - xo).max() < RTOL * np.abs(xo).max()


@pytest.mark.gpu
@pytest.mark.parametrize("ch,n,n_fft,hop", ROWS_REGRESSION + ROWS_SEAMS)
def test_rows_path_blocks(ch, n, n_fft, hop):
    """Batches the rows planner cuts into blocks of frames or of channels (and, for the first two, batches whose rows
    did not fit one launch): the first and last channel of every channel block equal the one-channel call, and
    frames on both sides of every frame seam agree with the oracle; stft and istft likewise."""
    import torch
    nfr = n_frames(n, hop)
    M, rows_max, blocks = rows_plan(n_fft, ch, nfr)
    assert len(blocks) >= 2
    pow2 = n_fft & (n_fft - 1) == 0
    kernel = "fft_pass rows + stft_generic_kernel<rows>"
    if not pow2:
        kernel = "bluestein " + kernel
    eng = _engine()
    x = _signals(ch, n, 11 + n_fft)
    win = np.hanning(n_fft)
    extra = {c for c0, cc, _, _ in blocks for c in (c0, c0 + cc - 1)}
    sampled = _sampled(ch, (n_fft // 2 + 1) * nfr, extra)
    seams = sorted({f0 for _, _, f0, _ in blocks if f0 > 0})
    whole = nfr * n_fft <= 4_000_000  # small enough for the oracle on the whole channel
    slices_of = (lambda c: None) if whole else (lambda c: _stft_slices(nfr, hop, n_fft, blocks_f0=seams, span=32))
    Sx = _ssq_stft_family(eng, x, win, n_fft, hop, 1000.0, sampled, slices_of, kernel)
    xr = eng.istft(Sx, win, n_fft, hop, N=n)
    torch.cuda.synchronize()
    assert "istft_ola_kernel<rows>" in eng.last_kernel_name(), eng.last_kernel_name()
    for c in sampled:
        _istft_vs_oracle(xr[c], Sx[c], win, n_fft, hop, n)
        # tiles restart at every frame block, whose length differs between the batch and the one-channel call
        _istft_same(eng.istft(Sx[c:c + 1], win, n_fft, hop, N=n)[0], xr[c], False, n_fft, hop)
    del Sx, xr, x, eng
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# CWT family on the C3 ring block (4 channels x 2^20 samples x 576 scales) and 8-channel components
# ---------------------------------------------------------------------------------------------------------------------
def _close_by_abs_sum(got, ref, abs_ref, terms):
    """|got - ref| <= 2 (terms + 2) eps32 * abs_ref elementwise: the rounding of an fp32 sum of `terms` products,
    abs_ref being the same reference evaluated on |Re Tx| (a sum of absolute values)."""
    got = np.asarray(got, np.float64)
    lim = 2 * (terms + 2) * EPS32 * np.asarray(abs_ref, np.float64) + 1e-30
    bad = np.abs(got - ref) > lim
    assert not bad.any(), (int(bad.sum()), float(np.abs(got - ref).max()), float(lim.max()))


@pytest.mark.gpu
def test_cwt_and_ssq_cwt_on_the_c3_ring_block():
    """cwt (W, dW) and ssq_cwt of 4 channels x 2^20 samples x 576 scales (each map 2.42e9 elements): every channel
    equals the one-channel call (W, dW, the unfused ssq_cwt bit for bit; the fused tail's bins, and its Tx within
    1e-5 of each row's maximum), and rows of W, dW at the smallest, middle and largest scales agree with the oracle."""
    import torch
    ch, n = 4, 1 << 20
    eng = _engine()
    sc = eng.default_scales(n, 32)
    assert len(sc) == 576 and ch * 576 * n > 1 << 31
    _free_and_need(2 * ch * 576 * n * 8 + (8 << 30))
    x = _signals(ch, n, 3)
    W, dW = eng.cwt(x, "gmw", sc, derivative=True)
    torch.cuda.synchronize()
    assert eng.last_kernel_name() == "fft_pass_kernel"
    rows = [0, 1, 287, 574, 575]
    for c in range(ch):
        Wc, dWc = eng.cwt(x[c:c + 1], "gmw", sc, derivative=True)
        assert torch.equal(Wc[0], W[c]) and torch.equal(dWc[0], dW[c]), c
        Wo, _, dWo = O.cwt(x[c].cpu().numpy().astype(np.float64), "gmw", sc[rows], derivative=True)
        ri = torch.as_tensor(rows, device="cuda")
        for got, ref in ((W[c][ri], Wo), (dW[c][ri], dWo)):
            got = got.cpu().numpy().astype(np.complex128)
            assert np.abs(got - ref).max() < RTOL * np.abs(ref).max(), c
    del W, dW, Wc, dWc
    torch.cuda.empty_cache()
    Tx, _, aux = eng.ssq_cwt(x, "gmw", sc, return_aux=True)
    torch.cuda.synchronize()
    assert "fused" in eng.last_kernel_name(), eng.last_kernel_name()
    kb = aux["kb"]
    del aux
    for c in range(ch):
        Tc, _, ac = eng.ssq_cwt(x[c:c + 1], "gmw", sc, return_aux=True)
        assert torch.equal(ac["kb"][0], kb[c]), c
        lim = 1e-5 * Tc[0].abs().amax(dim=1, keepdim=True)
        assert bool(((Tx[c] - Tc[0]).abs() <= lim).all()), c
        del Tc, ac
    del Tx
    torch.cuda.empty_cache()
    eng.ctx.set_option("no_cwt_fused", 1)
    try:
        Tn, _, an = eng.ssq_cwt(x, "gmw", sc, return_aux=True)
        torch.cuda.synchronize()
        assert "reassign" in eng.last_kernel_name(), eng.last_kernel_name()
        assert torch.equal(an["kb"], kb)  # same W, dW bits -> same bins as the fused tail
        del an, kb
        for c in range(ch):
            assert torch.equal(eng.ssq_cwt(x[c:c + 1], "gmw", sc)[0], Tn[c]), c
    finally:
        eng.ctx.set_option("no_cwt_fused", 0)
    del Tn, x, eng
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_inversions_and_components_past_2_31():
    """8 channels x 576 scales x 2^20 (38.7 GB maps): icwt of W, issq_cwt of Tx in full and in curve bands, and
    issq_stft bands of the same map read as 576 STFT rows; channels 0, 3 (element 2^31) and 7 (2^32) equal the
    one-channel call and agree with the float64 references on column slices."""
    import torch
    from test_components import stft_components
    ch, n = 8, 1 << 20
    eng = _engine()
    sc = eng.default_scales(n, 32)
    ns = len(sc)
    _free_and_need(ch * ns * n * 8 + (8 << 30))
    x = _signals(ch, n, 5)
    sampled = _sampled(ch, ns * n)
    assert sampled == [0, 3, 7]
    cols = [slice(0, 384), slice(n // 2 - 100, n // 2 + 100), slice(n - 384, n)]

    W = eng.cwt(x, "gmw", sc)
    xr = eng.icwt(W, sc, "gmw")
    torch.cuda.synchronize()
    assert eng.last_kernel_name() == "icwt_kernel"
    for c in sampled:
        assert torch.equal(eng.icwt(W[c:c + 1], sc, "gmw")[0], xr[c]), c
        for s in cols:
            Wh = W[c][:, s].cpu().numpy().astype(np.complex128)
            _close_by_abs_sum(xr[c][s].cpu().numpy(), O.icwt(Wh, "gmw", sc),
                              np.abs(O.icwt(np.abs(Wh.real) + 0j, "gmw", sc)), ns)
    del W, xr
    torch.cuda.empty_cache()

    Tx = eng.ssq_cwt(x, "gmw", sc)
    g = torch.Generator(device="cuda")
    g.manual_seed(17)
    K = 2
    cc = torch.randint(-1, ns, (ch, n, K), generator=g, device="cuda", dtype=torch.int32)
    cw = torch.randint(0, 9, (ch, n, K), generator=g, device="cuda", dtype=torch.int32)
    xs = eng.issq_cwt(Tx, sc, "gmw")
    assert eng.last_kernel_name() == "icwt_kernel"
    comp = eng.issq_cwt(Tx, sc, "gmw", cc=cc, cw=cw)
    assert eng.last_kernel_name() == "issq_components_kernel"
    nf = 2 * (ns - 1)
    win = np.hanning(nf)
    ycomp = eng.issq_stft(Tx, win, nf, 1.0, cc=cc, cw=cw)
    assert eng.last_kernel_name() == "issq_components_kernel"
    torch.cuda.synchronize()
    for c in sampled:
        one = (Tx[c:c + 1], cc[c:c + 1], cw[c:c + 1])
        assert torch.equal(eng.issq_cwt(one[0], sc, "gmw")[0], xs[c]), c
        assert torch.equal(eng.issq_cwt(one[0], sc, "gmw", cc=one[1], cw=one[2])[0], comp[c]), c
        assert torch.equal(eng.issq_stft(one[0], win, nf, 1.0, cc=one[1], cw=one[2])[0], ycomp[c]), c
        for s in cols:
            Th = Tx[c][:, s].cpu().numpy().astype(np.complex128)
            Ta = np.abs(Th.real) + 0j
            cch, cwh = cc[c][s].cpu().numpy(), cw[c][s].cpu().numpy()
            _close_by_abs_sum(xs[c][s].cpu().numpy(), O.issq_cwt(Th, "gmw", sc), O.issq_cwt(Ta, "gmw", sc), ns)
            _close_by_abs_sum(comp[c][:, s].cpu().numpy(), O.issq_cwt(Th, "gmw", sc, cch, cwh),
                              O.issq_cwt(Ta, "gmw", sc, cch, cwh), ns)
            _close_by_abs_sum(ycomp[c][:, s].cpu().numpy(), stft_components(Th, win, nf, 1.0, cch, cwh),
                              stft_components(Ta, win, nf, 1.0, cch, cwh), ns)
    del Tx, xs, comp, ycomp, cc, cw, x, eng
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# ridge extraction: many rows, and channel batches
# ---------------------------------------------------------------------------------------------------------------------
def _ridge_map(F, Tn, seed, dtype):
    """Noise under two drifting ridges: rows not a multiple of 4 and time steps not a multiple of TT are the callers'."""
    rng = np.random.default_rng(seed)
    Tf = rng.standard_normal((F, Tn)) + 1j * rng.standard_normal((F, Tn))
    t = np.arange(Tn)
    for r0, dr in ((F // 5, 3), (3 * F // 4, -2)):
        Tf[np.clip(r0 + dr * t + rng.integers(-2, 3, Tn), 0, F - 1), t] += 12.0
    return Tf.astype(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("F,dtype", [(F, np.complex64) for F, _ in RIDGE_ROWS_F32] + [(1025, np.complex128),
                                                                                   (5113, np.complex128)])
def test_ridges_many_rows_against_the_oracle(F, dtype):
    """Every time tile of ridge_run's rule (TT = 32 .. 1 in float, TT = 1 at double's limit of 5113 rows), rows above
    1024 (the kernels loop over f): the device's dynamic programme equals the oracle's bit for bit given the device's
    E (`_device_vs_oracle`)."""
    from ssqueeze_rs_b200 import _lib
    from test_ridges import _device_vs_oracle
    Tn = 37 if F <= 2047 else 13
    itemsize = 8 if dtype == np.complex128 else 4
    TT = ridge_plan(F, Tn, 1, itemsize)[0]
    assert Tn % TT or TT == 1
    Tf = _ridge_map(F, Tn, F, dtype)
    sc = 2.0 ** np.linspace(1, 9, F)
    _device_vs_oracle(Tf, sc, penalty=0.5, n_ridges=2 if F <= 2047 else 1, bw=4, transform="cwt")
    assert _lib.default_context().last_kernel_name() == "ridge_forward_kernel"


@pytest.mark.gpu
def test_ridges_double_above_its_row_limit_is_unsupported():
    """Two [F][2] tiles of float64 do not fit 200 KiB of shared memory above 5113 rows: a clean SSQ_EUNSUPPORTED that
    names the limit, and nothing launched."""
    import ctypes as C
    from ssqueeze_rs_b200 import _lib
    ctx = _lib.default_context()
    F, Tn = ridge_rows_limit(8) + 1, 5
    Tf = _ridge_map(F, Tn, 1, np.complex128)
    sc = 2.0 ** np.linspace(1, 9, F)
    idx = np.empty((Tn, 1), np.int32)
    st = _lib.load().ssq_extract_ridges_host(ctx.handle, C.c_void_p(Tf.ctypes.data), 1, F, Tn,
                                            C.c_void_p(sc.ctypes.data), 2.0, 1, 4, 0, C.c_void_p(idx.ctypes.data),
                                            C.c_void_p(0), C.c_void_p(0), C.c_void_p(0))
    assert st == SSQ_EUNSUPPORTED
    msg = _lib.load().ssq_last_error(ctx.handle).decode()
    assert "5114" in msg and "5113" in msg, msg
    # the float map of the same rows runs
    from ssqueeze_rs_b200 import _rs
    _rs.extract_ridges(Tf.astype(np.complex64), sc, n_ridges=1, bw=4)


@pytest.mark.gpu
def test_ridges_channel_batches():
    """373 channels of 257 x 56 250 (the C2 map, 43 GB in complex64): ridge_run's 20 GiB channel batches hold 371
    channels, so channels 370 | 371 straddle the batch seam; those, the first and the last equal the one-channel call
    bit for bit (indices, ridge_f, ridge_e)."""
    import torch
    ch, F, Tn = RIDGE_BATCH
    TT, cb = ridge_plan(F, Tn, ch, 4)
    assert cb == 371
    _free_and_need(ch * F * Tn * 8 + 3 * cb * F * Tn * 4 + (2 << 30))
    eng = _engine()
    Tf = torch.empty((ch, F, Tn), dtype=torch.complex64, device="cuda")
    g = torch.Generator(device="cuda")
    t = torch.arange(Tn, device="cuda")
    for c in range(ch):
        g.manual_seed(2_000_003 + c)
        Tf[c] = torch.randn((F, Tn), generator=g, device="cuda", dtype=torch.complex64)
        Tf[c, (10 + c % 200 + (t // 5000)) % F, t] += 10.0
    sc = 2.0 ** np.linspace(1, 8, F)
    kw = dict(penalty=2.0, n_ridges=2, bw=4, transform="cwt", get_params=True)
    idx, rf, re_ = eng.extract_ridges(Tf, sc, **kw)
    torch.cuda.synchronize()
    assert eng.last_kernel_name() == "ridge_forward_kernel"
    for c in (0, cb - 1, cb, ch - 1):
        i1, f1, e1 = eng.extract_ridges(Tf[c:c + 1], sc, **kw)
        assert torch.equal(i1[0], idx[c]) and torch.equal(f1[0], rf[c]) and torch.equal(e1[0], re_[c]), c
        # the strong ridge of channel c is found (a swapped channel would not be)
        assert float((idx[c, :, 0] == (10 + c % 200 + t // 5000) % F).float().mean()) > 0.9, c
    del Tf, idx, rf, re_, eng
    gc.collect()
    torch.cuda.empty_cache()

"""GPU: the CWT streams (ssq_stream_create_cwt, CwtStream; DESIGN §3.6b).  Block b of a stream is the batch call on
its materialised extended input x~[bC - d, bC + len_b + d), trimmed to columns [d, d + len_b): bit for bit for cwt
and for ssq_cwt on the stand-alone reassignment, up to the order of the float additions into Tx on the fused path.
The output does not depend on how the recording is cut into pushes."""
import ctypes as C

import numpy as np
import pytest

from oracle import cwt_blocks as B
from oracle import parity as P
from oracle import ssq_oracle as O

pytestmark = pytest.mark.gpu
FS = 1000.0
FUSED_RTOL = 1e-5  # fused Tx: atomics from several CTAs add into one element in no fixed order


def _rec(N, channels, dtype, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(N) / FS
    base = np.sin(2 * np.pi * (5 * t + 40 * t * t / max(t[-1], 1e-3)))[:, None] * 800
    noise = rng.standard_normal((N, channels)) * 300
    if dtype == "i16":
        return np.clip(base + noise, -32000, 32000).astype(np.int16), 0.195
    return ((base + noise) / 100).astype(np.float32), 1.0


def _materialised(eng, rec, scale, C_, d, transform, scales, **kw):
    """The batch call on the extended blocks of every channel, one call per block length, trimmed and laid out as the
    stream lays out its columns; also the ssq grid of each call."""
    import torch
    N, ch = rec.shape
    x = rec.astype(np.float32) * np.float32(scale)
    nb = B.n_blocks(N, C_)
    groups = [list(range(nb))] if N % C_ == 0 else [list(range(nb - 1)), [nb - 1]]
    outs, freqs = [], []
    for g in groups:
        if not g:
            continue
        ln = B.block_len(N, C_, g[0])
        e = np.stack([B.extended_block(x, C_, d, b) for b in g], axis=0)  # [nb, e_len, ch]
        xt = torch.from_numpy(np.ascontiguousarray(e.transpose(2, 0, 1).reshape(ch * len(g), -1))).cuda()
        if transform == "cwt":
            W = eng.cwt(xt, scales=scales, fs=FS, **kw)
            sf = None
        else:
            W, sf = eng.ssq_cwt(xt, scales=scales, fs=FS, return_freqs=True, **kw)
        W = W[:, :, d:d + ln].reshape(ch, len(g), len(scales), ln).permute(0, 2, 1, 3).reshape(ch, len(scales), -1)
        outs.append(W)
        freqs.append(sf)
    return torch.cat(outs, dim=2), freqs


def _stream(eng, rec, scale, C_, d, pushes, transform, scales, **kw):
    import torch
    from ssqueeze_rs_b200.batch import CwtStream
    N, ch = rec.shape
    st = CwtStream(eng, ch, N, max(pushes), C_, d, scales=scales, fs=FS, transform=transform, **kw)
    assert st.total_frames == N
    parts, pos, i = [], 0, 0
    while pos < N:
        c = min(pushes[i % len(pushes)], N - pos)
        parts.append(st.push(torch.from_numpy(np.ascontiguousarray(rec[pos:pos + c])).cuda(), scale))
        pos += c
        i += 1
    got = torch.cat(parts, dim=2)
    grids = (st.ssq_freqs(), st.ssq_freqs(last=True)) if transform == "ssq_cwt" else None
    st.close()
    return got, grids


def _check(N, C_, d, pushes, transform="ssq_cwt", channels=2, dtype="f32", fused=None, nsc=10, expect=None, **kw):
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    rec, scale = _rec(N, channels, dtype, N + C_ + d)
    scales = 2.0 ** np.linspace(1, np.log2(max(C_ + 2 * d, 8) / 4), nsc)
    if fused is not None:
        eng.ctx.set_option("no_cwt_fused", 0 if fused else 1)
    try:
        ref, freqs = _materialised(eng, rec, scale, C_, d, transform, scales, **kw)
        one, grids = _stream(eng, rec, scale, C_, d, [N], transform, scales, **kw)
        name = eng.last_kernel_name()
        rag, _ = _stream(eng, rec, scale, C_, d, pushes, transform, scales, **kw)
    finally:
        eng.ctx.set_option("no_cwt_fused", 0)
    torch.cuda.synchronize()
    assert one.shape == ref.shape == (channels, nsc, N)
    exact = transform == "cwt" or fused is False
    if expect is not None:
        assert expect in name, name
    if exact:
        assert torch.equal(one, ref), float((one - ref).abs().max())
        assert torch.equal(rag, one), float((rag - one).abs().max())
    else:
        tol = FUSED_RTOL * float(ref.abs().max())
        assert float((one - ref).abs().max()) <= tol
        assert float((rag - one).abs().max()) <= tol
    if grids is not None:
        assert np.array_equal(grids[0], freqs[0]) if N >= C_ else True
        assert np.array_equal(grids[1], freqs[-1])
    return name


# L of the extended blocks (the last, shorter block's too): 2^14 and 2^18 end in a 7-bit register pass (fused
# ssq_cwt), 2^13 and 2^15 do not
@pytest.mark.parametrize("N,C_,d,L,fused", [(22000, 6000, 1000, 14, True), (250000, 100000, 20000, 18, True),
                                            (9000, 2000, 500, 13, False), (40000, 15000, 2000, 15, False)])
def test_plans(N, C_, d, L, fused):
    e = C_ + 2 * d
    assert O.next_power_of_2(e + e // 2) == 1 << L
    pushes = [1, d // 2 + 3, 3 * C_ + 17, 777]
    _check(N, C_, d, pushes, "cwt")
    name = _check(N, C_, d, pushes, "ssq_cwt", maprange="maximal")
    assert ("fused" in name) == fused, name
    if fused:
        _check(N, C_, d, pushes, "ssq_cwt", fused=False, expect="reassign", maprange="maximal")


@pytest.mark.parametrize("N,C_,d", [(20000, 6000, 0), (9000, 2000, 2000), (3000, 5000, 1000), (1500, 2000, 1500),
                                    (7001, 7001, 100), (1, 1, 1)])
def test_geometries(N, C_, d):
    """d = 0; d = C with a last block (1000) shorter than d; N < C (one block); N = d; one block exactly; N = 1."""
    pushes = [max(1, d // 3), 1, 2 * C_ + 1]
    for transform in ("cwt", "ssq_cwt"):
        _check(N, C_, d, pushes, transform, fused=False, nsc=6 if N > 1 else 1)
        _check(N, C_, d, pushes, transform, nsc=6 if N > 1 else 1)


@pytest.mark.parametrize("kw", [dict(dtype="i16"), dict(wavelet="morlet"), dict(maprange="maximal"),
                                dict(padtype="zero"), dict(squeezing="lebesgue"), dict(flipud=False),
                                dict(ssq_freqs="linear", maprange="maximal"), dict(gamma=0.5), dict(channels=5)])
def test_ssq_cwt_options(kw):
    kw = dict(kw)
    for fused in (False, True):
        _check(30000, 7000, 1500, [4096, 1, 999], "ssq_cwt", fused=fused, **kw)


@pytest.mark.parametrize("kw", [dict(l1_norm=False), dict(wavelet="morlet", dtype="i16"), dict(padtype="zero")])
def test_cwt_options(kw):
    _check(30000, 7000, 1500, [4096, 1, 999], "cwt", channels=3, **kw)


def test_default_scales_and_last_block_grid():
    import torch
    from ssqueeze_rs_b200.batch import CwtStream, Engine
    eng = Engine(0)
    st = CwtStream(eng, 1, 10000, 10000, 3000, 500, fs=FS, nv=8, maprange="maximal")
    assert np.array_equal(st.scales, eng.default_scales(4000, 8))
    full, last = st.ssq_freqs(), st.ssq_freqs(last=True)
    assert np.isclose(full[0], FS / 4000) and np.isclose(last[0], FS / 2000)  # 1000 + 2 * 500 samples
    out = st.push(torch.zeros((10000, 1), dtype=torch.float32, device="cuda"))
    assert out.shape == (1, len(st.scales), 10000)
    st.close()


def _write_recordings(tmp_path, rec):
    import pyarrow as pa
    import pyarrow.parquet as pq
    path = tmp_path / "rec.dat"
    rec.tofile(path)
    pq.write_table(pa.table({f"c{i}": rec[:, i] for i in range(rec.shape[1])}), tmp_path / "rec.parquet")
    return np.memmap(path, dtype=rec.dtype, mode="r").reshape(-1, rec.shape[1]), tmp_path / "rec.parquet"


@pytest.mark.parametrize("transform", ["ssq_cwt", "cwt"])
def test_feeder_drives_the_stream(tmp_path, transform):
    """RecordingFeeder(stream=...) from a memory-mapped int16 file and from ParquetRecording: the direct pushes."""
    import torch
    from ssqueeze_rs_b200.batch import CwtStream, Engine, ParquetRecording, RecordingFeeder
    eng = Engine(0)
    N, ch, C_, d = 50000, 4, 9000, 2000
    rec, scale = _rec(N, ch, "i16", 11)
    mm, pq_path = _write_recordings(tmp_path, rec)
    sc = 2.0 ** np.linspace(1, 9, 12)
    direct, _ = _stream(eng, rec, scale, C_, d, [6000], transform, sc)
    for src in (mm, ParquetRecording(pq_path, batch_rows=5000)):
        st = CwtStream(eng, ch, N, 6000, C_, d, scales=sc, fs=FS, transform=transform)
        with RecordingFeeder(eng, src, None, chunk=1 << 20, scale=scale, stream=st) as feed:
            assert feed.chunk == 6000
            got = torch.cat(list(feed), dim=2)
        torch.cuda.synchronize()
        st.close()
        if transform == "cwt":
            assert torch.equal(got, direct)
        else:
            assert float((got - direct).abs().max()) <= FUSED_RTOL * float(direct.abs().max())


def test_against_the_float64_oracle():
    """Wx within the CWT tolerance of the blockwise float64 oracle; every bin of the materialised-block ssq_cwt call
    classified with nothing unexplained, and the stream equal to that call."""
    import torch
    from ssqueeze_rs_b200.batch import CwtStream, Engine
    eng = Engine(0)
    N, C_, d = 3000, 1000, 300
    x = _rec(N, 1, "f32", 3)[0][:, 0].astype(np.float64)
    sc = 2.0 ** np.linspace(1, 7, 12)
    st = CwtStream(eng, 1, N, N, C_, d, scales=sc, fs=FS, transform="cwt")
    W = st.push(torch.from_numpy(x.astype(np.float32)[:, None].copy()).cuda())[0].cpu().numpy()
    st.close()
    Wo = B.blockwise_cwt(x, C_, d, sc, fs=FS)
    assert np.abs(W - Wo).max() / np.abs(Wo).max() < 1e-4
    st = CwtStream(eng, 1, N, N, C_, d, scales=sc, fs=FS, maprange="maximal")
    T = st.push(torch.from_numpy(x.astype(np.float32)[:, None].copy()).cuda())[0]
    st.close()
    for b in range(B.n_blocks(N, C_)):
        e = B.extended_block(x, C_, d, b)
        Tb, sf, aux = eng.ssq_cwt(torch.from_numpy(e.astype(np.float32)[None]).cuda(), scales=sc, fs=FS,
                                  maprange="maximal", return_aux=True)
        To, sfo, ao = O.ssq_cwt(e.astype(np.float32).astype(np.float64), scales=sc, fs=FS, maprange="maximal",
                                return_aux=True)
        rep = P.classify_cwt_bins(aux["kb"][0].cpu().numpy(), ao, e.astype(np.float32).astype(np.float64), "gmw",
                                  1.0 / FS, "reflect", sfo, w_dev=aux["w"][0].cpu().numpy())
        assert rep["unexplained"] == 0, P.public(rep)
        assert torch.equal(T[:, b * C_:(b + 1) * C_], Tb[0, :, d:d + C_])


def test_argument_errors_leave_no_stream():
    from ssqueeze_rs_b200 import _lib
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    sc = np.array([2.0, 4.0])
    lib = _lib.load()

    def create(n_total=1000, block=100, overlap=10, mode=3, ns=2):
        h = C.c_void_p(123)
        st = lib.ssq_stream_create_cwt(eng.ctx.handle, 1, n_total, 100, block, overlap, mode, 0,
                                       C.c_void_p(sc.ctypes.data), ns, 1.0, 0, 0, 0, 0, float("nan"), 0, C.byref(h))
        return st, h.value

    for kw in (dict(block=0), dict(overlap=101), dict(overlap=-1), dict(n_total=5, block=10, overlap=6), dict(ns=0),
               dict(mode=1), dict(mode=4)):
        st, h = create(**kw)
        assert st == 1 and h is None, kw  # SSQ_EINVAL
    st, h = create()
    assert st == 0 and h
    lib.ssq_stream_destroy(C.c_void_p(h))

"""The n_fft 512 ssq kernel keeps its window taps, and at hop 32 its sliding sample window, in tensor memory
(tcgen05.ld / st).  Every instantiation of the ssq mode -- hop 32 and any other hop, both squeezings, the diagnostic
variant -- must give the Tx it gave with the taps in a shared-memory table and the samples in registers, bit for bit:
the multiplications take the same fp32 operands.

tests/golden/h32r_tx_sha256.json holds the SHA-256 of the complex64 Tx of each case below as computed by the kernel
before the change (`python tests/test_h32r_tmem.py --write-golden` writes it).  Each case also checks the destination
bins against the generic shared-memory kernel (`no_h32r`), an independent implementation.

Cases: edge tiles under reflect and zero padding with a ragged last tile, hop != 32, Lebesgue squeezing, a tonal
signal (the collision paths), more tiles than resident CTAs (every CTA runs several tiles), and two contexts on two
streams launched back to back."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "h32r_tx_sha256.json")
FS = 30000.0
KERNEL = "ssq_stft512_h32r_kernel<ssq>"

# name -> (signal, channels, samples, hop, options)
CASES = {
    "reflect_hop32": ("noise_tone", 2, 1500, 32, {}),  # 47 frames: edge tiles at both ends, last tile 15 of 16
    "zero_hop32": ("noise_tone", 2, 1500, 32, dict(padtype="zero")),
    "lebesgue_hop32": ("noise_tone", 2, 1500, 32, dict(squeezing="lebesgue")),
    "tone_hop32": ("tone", 1, 3001, 32, {}),
    "reflect_hop17": ("noise_tone", 2, 1500, 17, {}),  # 89 frames, per-frame sample reload
    "zero_hop48": ("noise", 3, 2000, 48, dict(padtype="zero")),
    "many_tiles_hop32": ("noise_tone", 64, 8000, 32, {}),  # 1 024 tiles: more than one per CTA on any GPU here
}


def signal(kind, channels, n):
    rng = np.random.default_rng(0x7E3 + channels * 7919 + n)
    t = np.arange(n) / FS
    tone = 50.0 * np.sin(2 * np.pi * 1234.5 * t) + 20.0 * np.sin(2 * np.pi * 7000.0 * t)
    if kind == "tone":
        x = np.tile(tone, (channels, 1))
    elif kind == "noise":
        x = 30.0 * rng.standard_normal((channels, n))
    else:
        x = tone + 10.0 * rng.standard_normal((channels, n))
    return np.ascontiguousarray(x, dtype=np.float32)


def digest(Tx):
    import torch
    assert Tx.dtype == torch.complex64
    return hashlib.sha256(Tx.contiguous().cpu().numpy().tobytes()).hexdigest()


def run(eng, name, aux=False):
    import torch
    kind, ch, n, hop, kw = CASES[name]
    x = torch.from_numpy(signal(kind, ch, n)).cuda()
    return eng.ssq_stft(x, np.hanning(512), 512, hop, FS, return_aux=aux, **kw)


def write_golden(path):
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    out = {}
    for name in CASES:
        Tx = run(eng, name)
        assert eng.last_kernel_name() == KERNEL, eng.last_kernel_name()
        out[name] = digest(Tx)
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN) as f:
        return json.load(f)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_tx_as_before_and_bins_as_generic(name, golden):
    import torch
    from ssqueeze_rs_b200.batch import Engine
    eng = Engine(0)
    Tx = run(eng, name)
    assert eng.last_kernel_name() == KERNEL
    assert digest(Tx) == golden[name]
    # the diagnostic variant (the same kernel with the aux stores compiled in) agrees bit for bit
    Tx_d, aux = run(eng, name, aux=True)
    assert eng.last_kernel_name() == KERNEL
    torch.cuda.synchronize()
    assert torch.equal(Tx_d, Tx)
    eng.ctx.set_option("no_h32r", 1)
    try:
        Tg, aux_g = run(eng, name, aux=True)
        assert "generic" in eng.last_kernel_name(), eng.last_kernel_name()
    finally:
        eng.ctx.set_option("no_h32r", 0)
    # the generic kernel's FFT rounds differently: a bin whose w sits on a bin edge may flip, nothing else differs.
    # Bins far below the frame's energy (the skirts of a pure tone) have an ill-conditioned w in either kernel and
    # are left to the oracle parity tests.
    mag = aux_g["Sx"].abs()
    strong = mag > 1e-3 * mag.amax(dim=1, keepdim=True)
    flips = float((aux["kb"] != aux_g["kb"])[strong].float().mean())
    assert flips < 2e-3, flips
    sc = float(Tg.abs().max())
    assert float((Tx.sum(dim=1) - Tg.sum(dim=1)).abs().max()) < 2e-3 * sc
    assert float(((Tx - Tg).abs() > 1e-4 * sc).float().mean()) < 2e-3


@pytest.mark.gpu
def test_two_contexts_two_streams_back_to_back(golden):
    """Two contexts on two streams, launched without a synchronisation between them: the CTAs of both launches share
    the SMs and each allocates its own tensor-memory columns."""
    import torch
    from ssqueeze_rs_b200.batch import Engine
    engs = [Engine(0), Engine(0)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    names = ["many_tiles_hop32", "reflect_hop17"]
    outs = []
    for _ in range(2):
        for eng, s, name in zip(engs, streams, names):
            with torch.cuda.stream(s):
                outs.append((name, run(eng, name)))
            assert eng.last_kernel_name() == KERNEL
    torch.cuda.synchronize()
    for name, Tx in outs:
        assert digest(Tx) == golden[name], name


if __name__ == "__main__":
    if sys.argv[1:2] != ["--write-golden"]:
        sys.exit("usage: python tests/test_h32r_tmem.py --write-golden [path]")
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    write_golden(sys.argv[2] if len(sys.argv) > 2 else GOLDEN)

"""bench.py's command line: --steps sets the number of timed steps, and --dump-outputs writes a seeded sample of the
timed step's Tx that is the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _bench(*args, timeout=60):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout)


@pytest.mark.parametrize("args", [["--steps", "0"],
                                  ["--impl", "reference", "--dump-outputs", "out"],
                                  ["--workload", "istft", "--dump-outputs", "out"],
                                  ["--n-fft", "1024", "--dump-outputs", "out"]])
def test_rejected_arguments(args, tmp_path):
    r = _bench(*[str(tmp_path / a) if a == "out" else a for a in args])
    assert r.returncode == 2 and "error" in r.stderr, r.stderr[-2000:]
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_and_steps(tmp_path):
    import torch
    import bench
    from ssqueeze_rs_b200.batch import Engine
    ch, n = 4, 200_000
    lines = {}
    for steps in (2, 3):
        r = _bench("--gpus", "1", "--steps", str(steps), "--warmup", "1", "--channels", str(ch), "--samples", str(n),
                   "--no-cpu-baseline", "--no-side-configs", "--dump-outputs", str(tmp_path / f"s{steps}"), timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        lines[steps] = json.loads(r.stdout.strip().splitlines()[-1])
        assert lines[steps]["steps"] == steps
    # the launches inside the timed region scale with --steps
    assert lines[2]["gpu_launches"] > 0 and lines[2]["gpu_launches"] * 3 == lines[3]["gpu_launches"] * 2
    a, b = (np.load(tmp_path / f"s{s}" / "Tx.npy") for s in (2, 3))
    nfr = (n - 1) // bench.HOP + 1
    k = min(bench.DUMP_COLUMNS, ch * nfr)
    assert a.dtype == np.float32 and a.shape == (k, bench.N_FFT // 2 + 1, 2) and a.nbytes <= 64 << 20
    assert np.array_equal(a, b)  # same arguments, same input, same output
    # the dump is the sampled columns of what the engine returns for the bench's input
    eng = Engine(0)
    x = bench.make_neural(torch, ch, n, bench.FS, torch.device("cuda", 0), 0x5351)
    Tx = eng.ssq_stft(x, np.hanning(bench.N_FFT), bench.N_FFT, bench.HOP, bench.FS).cpu().numpy()
    flat = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(ch * nfr, size=k, replace=False))
    cols = Tx[flat // nfr, :, flat % nfr]
    assert np.array_equal(a[..., 0], cols.real) and np.array_equal(a[..., 1], cols.imag)
    assert np.abs(cols).max() > 0

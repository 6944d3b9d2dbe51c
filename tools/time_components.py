"""Device time of the component inversion (`Engine.issq_cwt` / `Engine.issq_stft` with `cc`, `cw`; DESIGN §3.7) against
the full inversion on the same Tx.

Geometries (every Tx is larger than the 126 MB L2, so each call reads it from HBM):
  * CWT: 8 channels x 2^20 samples x 576 scales (Tx 38.7 GB), cc a seeded random walk over the rows, cw = 8, for
    K = 1, 2, 4, 16, against `Engine.issq_cwt(Tx, scales)`;
  * STFT: 16 channels x 2^20 frames, n_fft 512, hop 1 (Tx 34.5 GB), K = 1, 2, against `Engine.issq_stft`.
Tx is seeded noise: the kernels' work does not depend on its values.  Each call runs once as warm-up, then `--reps`
times between CUDA events; the best is reported, with GB/s over the bytes the call has to move,
8 n_rows n (Tx) + 8 K n (cc, cw) + 4 (K + 1) n (the result) per channel (the full inversion: 8 n_rows n + 4 n), and as
a share of the device-to-device copy bandwidth measured in the same run (a torch copy of `--copy-gb` GB: read + write).
The card's name and power limit are recorded with the numbers.

    python tools/time_components.py [--reps 3] [--json components.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still worth printing; say that the card was not identified
        q = f"nvidia-smi unavailable ({e})"
    return q


def best_ms(fn, reps):
    import torch
    ts = []
    for rep in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if rep:
            ts.append(e0.elapsed_time(e1))
    return min(ts)


def random_walk(ch, n, K, n_rows, seed):
    """int32 [ch, n, K]: K curves per channel, each a +-1 random walk over the rows from a random start, clipped."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    start = torch.randint(0, n_rows, (ch, 1, K), generator=g, device="cuda", dtype=torch.int64)
    steps = torch.randint(-1, 2, (ch, n, K), generator=g, device="cuda", dtype=torch.int64)
    return (start + steps.cumsum(1)).clamp_(0, n_rows - 1).to(torch.int32).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n", type=int, default=1 << 20, help="samples (CWT) / frames (STFT) per channel")
    ap.add_argument("--cwt-channels", type=int, default=8)
    ap.add_argument("--stft-channels", type=int, default=16)
    ap.add_argument("--copy-gb", type=float, default=8.0)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()

    import torch
    from ssqueeze_rs_b200.batch import Engine
    if not torch.cuda.is_available():
        raise SystemExit("time_components.py measures on a CUDA device; none is available")
    eng = Engine(0)
    n = a.n
    res = {"card": card(), "timing": f"CUDA events around the call, best of {a.reps} after one warm-up",
           "bytes": "8 n_rows n + 8 K n + 4 (K + 1) n per channel"}
    print(res["card"], flush=True)

    # device-to-device copy bandwidth (read + write)
    m = int(a.copy_gb * 1e9) // 4
    src = torch.empty(m, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    ms = best_ms(lambda: dst.copy_(src), a.reps)
    copy_gbs = 2 * m * 4 / (ms * 1e-3) / 1e9
    res["d2d_copy"] = {"GB": m * 4 / 1e9, "ms": ms, "GB_per_s": copy_gbs}
    print(f"d2d copy of {m * 4 / 1e9:.1f} GB: {ms:.3f} ms, {copy_gbs:.0f} GB/s (read + write)", flush=True)
    del src, dst
    torch.cuda.empty_cache()

    def record(key, name, ch, n_rows, K, ms):
        by = ch * (8 * n_rows * n + (8 * K * n + 4 * (K + 1) * n if K else 4 * n))
        gbs = by / (ms * 1e-3) / 1e9
        r = {"ms": ms, "GB": by / 1e9, "GB_per_s": gbs, "share_of_copy_bw": gbs / copy_gbs,
             "kernel": eng.last_kernel_name()}
        res[key][name] = r
        print(f"  {name:18s} {ms:9.3f} ms  {gbs:7.0f} GB/s  {100 * gbs / copy_gbs:5.1f} % of copy  ({r['kernel']})",
              flush=True)
        return r

    def series(key, ch, n_rows, Ks, comp, seed):
        for K in Ks:
            cc = random_walk(ch, n, K, n_rows, seed + K)
            cw = torch.full_like(cc, 8)
            r = record(key, f"K={K}", ch, n_rows, K, best_ms(lambda: comp(cc, cw), a.reps))
            r["vs_full"] = r["ms"] / res[key]["full"]["ms"]
            print(f"  {'':18s} {r['vs_full']:.3f} x the full inversion", flush=True)
            del cc, cw

    g = torch.Generator(device="cuda").manual_seed(0)
    # ---- CWT ----
    ch, ns = a.cwt_channels, 576
    sc = eng.default_scales(n, 32)
    assert len(sc) == ns
    Tx = torch.randn((ch, ns, n), dtype=torch.complex64, device="cuda", generator=g)
    res["cwt"] = {"geometry": f"{ch} ch x {n} samples x {ns} scales, cw = 8", "Tx_GB": Tx.numel() * 8 / 1e9}
    print(f"cwt: {res['cwt']['geometry']}, Tx {res['cwt']['Tx_GB']:.1f} GB", flush=True)
    record("cwt", "full", ch, ns, 0, best_ms(lambda: eng.issq_cwt(Tx, sc), a.reps))
    series("cwt", ch, ns, (1, 2, 4, 16), lambda cc, cw: eng.issq_cwt(Tx, sc, cc=cc, cw=cw), 10)
    del Tx
    torch.cuda.empty_cache()

    # ---- STFT ----
    ch, nf = a.stft_channels, 512
    win = np.hanning(nf)
    Tx = torch.randn((ch, nf // 2 + 1, n), dtype=torch.complex64, device="cuda", generator=g)
    res["stft"] = {"geometry": f"{ch} ch x {n} frames, n_fft {nf}, hop 1, cw = 8", "Tx_GB": Tx.numel() * 8 / 1e9}
    print(f"stft: {res['stft']['geometry']}, Tx {res['stft']['Tx_GB']:.1f} GB", flush=True)
    record("stft", "full", ch, nf // 2 + 1, 0, best_ms(lambda: eng.issq_stft(Tx, win, nf), a.reps))
    series("stft", ch, nf // 2 + 1, (1, 2), lambda cc, cw: eng.issq_stft(Tx, win, nf, cc=cc, cw=cw), 20)
    del Tx
    torch.cuda.empty_cache()
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

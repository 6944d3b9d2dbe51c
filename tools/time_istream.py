"""Device time of the streaming inverse (`IstftStream`, DESIGN §3.4c) against the batch `Engine.istft` on the whole Sx,
and of the forward-stream -> inverse-stream round trip.

Default geometry: 384 channels x 1.8 M samples at n_fft 512 / hop 32 (Sx is 44.4 GB, so it fits on one B200 beside the
batch call's accumulator).  The batch call is timed with CUDA events around the call; the stream with CUDA events
around every push, summed over the pushes (the host gaps between pushes are not counted).  Each configuration runs
once as warm-up, then `--reps` times; the best and the median are reported as Msamples/s = channels x samples / time.
The stream's output is checked against the batch call's (max |diff| / max |x|).

    python tools/time_istream.py [--channels 384] [--samples 1800000] [--pushes 2048,8192,56250] [--json out.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=384)
    ap.add_argument("--samples", type=int, default=1_800_000)
    ap.add_argument("--pushes", default="2048,8192,56250", help="frames per push of the inverse stream")
    ap.add_argument("--rt-chunk", type=int, default=8192 * 32, help="samples per push of the round trip")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()

    import torch
    from ssqueeze_rs_b200.batch import Engine, IstftStream, SsqStftStream
    if not torch.cuda.is_available():
        raise SystemExit("time_istream.py measures on a CUDA device; none is available")
    N_FFT, HOP = 512, 32
    ch, n = a.channels, a.samples
    nfr = (n - 1) // HOP + 1
    eng = Engine(0)
    eng._bind_stream()
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn((ch, n), generator=g, device="cuda") * 20
    win = np.hanning(N_FFT)
    Sx = eng.stft(x, win, N_FFT, HOP)
    torch.cuda.synchronize()
    res = {"card": card(), "geometry": f"{ch} ch x {n} samples, n_fft {N_FFT} hop {HOP}, {nfr} frames",
           "Sx_GB": Sx.numel() * 8 / 1e9, "timing": "CUDA events; stream: summed over pushes"}
    print(res["card"], "|", res["geometry"], f"| Sx {res['Sx_GB']:.1f} GB", flush=True)

    def rate(ms):
        return ch * n / (ms * 1e-3) / 1e6

    def summary(name, ts, extra=None):
        ts = sorted(ts)
        r = {"best_ms": ts[0], "median_ms": ts[len(ts) // 2], "best_Msamples_per_s": rate(ts[0]),
             "median_Msamples_per_s": rate(ts[len(ts) // 2])}
        r.update(extra or {})
        res[name] = r
        print(f"{name:28s} best {ts[0]:9.2f} ms  median {r['median_ms']:9.2f} ms  {r['best_Msamples_per_s']:9.0f} "
              f"Msamples/s" + "".join(f"  {k} {v}" for k, v in (extra or {}).items()), flush=True)

    # ---- batch ----
    xb = torch.empty((ch, n), dtype=torch.float32, device="cuda")
    ts = []
    for rep in range(a.reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.istft(Sx, win, N_FFT, HOP, N=n, out=xb)
        e1.record()
        torch.cuda.synchronize()
        if rep:
            ts.append(e0.elapsed_time(e1))
    summary("batch istft", ts, {"kernel": eng.last_kernel_name()})
    xmax = float(xb.abs().max())

    # ---- stream, pushes of P frames ----
    for P in [int(p) for p in a.pushes.split(",")]:
        chunks = [Sx] if P >= nfr else [Sx[:, :, f:f + P].contiguous() for f in range(0, nfr, P)]
        ts, err = [], 0.0
        for rep in range(a.reps + 1):
            inv = IstftStream(eng, ch, nfr, min(P, nfr), win, N_FFT, HOP, N=n)
            total, pos = 0.0, 0
            for c in chunks:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                y = inv.push(c)
                e1.record()
                e1.synchronize()
                total += e0.elapsed_time(e1)
                if rep == 0:
                    err = max(err, float((y - xb[:, pos:pos + y.shape[1]]).abs().max()) / xmax)
                pos += y.shape[1]
                del y
            assert pos == n
            inv.close()
            if rep:
                ts.append(total)
        summary(f"stream istft, {P} frames", ts, {"pushes": len(chunks), "max_rel_diff_vs_batch": f"{err:.2e}"})
        del chunks
        torch.cuda.empty_cache()

    # ---- round trip: forward stft stream -> inverse stream ----
    del xb
    Sx = None
    torch.cuda.empty_cache()
    xi = x.t().contiguous()  # interleaved [samples, channels], as a recording arrives
    C = a.rt_chunk
    max_frames = (C + N_FFT) // HOP + 2
    ts = []
    for rep in range(a.reps + 1):
        fwd = SsqStftStream(eng, ch, n, C, win, N_FFT, HOP, transform="stft")
        inv = IstftStream(eng, ch, nfr, max_frames, win, N_FFT, HOP, N=n)
        total, pos, done = 0.0, 0, 0
        while pos < n:
            k = min(C, n - pos)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            y = inv.push(fwd.push(xi[pos:pos + k]))
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
            done += y.shape[1]
            pos += k
            del y
        assert done == n
        fwd.close()
        inv.close()
        if rep:
            ts.append(total)
    summary(f"round trip, {C} samples", ts, {"pushes": (n + C - 1) // C})
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

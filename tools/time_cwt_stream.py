"""Time the CWT stream (`CwtStream` driven by `RecordingFeeder`, DESIGN §3.6b) on a memory-mapped int16 recording.

Default: 64 channels x 2^22 int16 samples in a temporary file, GMW, nv 32, Tx reduced on the device after every push
(|Tx| summed over time per channel and row), in two geometries:
  - block 2^17, overlap 2^14: L = 2^18, the fused ssq_cwt path (Tx of one block for 64 channels is about 33 GB);
  - block 2^14, overlap 2^12: L = 2^16, the stand-alone reassignment.
Reported per geometry:
  - the feeder pass in Msamples/s = channels x samples / wall time of the pass (ends in a device synchronise);
  - the device time of the pushes, from CUDA events around each push on the compute stream, summed.  It includes any
    wait for the chunk's host-to-device copy;
  - the batch call on the materialised extended blocks of --ref-blocks full blocks (the same FFT work per block),
    timed with CUDA events, set against the stream's time per block.
The card name and power limit are printed with the numbers.

    python tools/time_cwt_stream.py [--channels 64] [--log2n 22] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still worth printing; say that the card was not identified
        q = f"nvidia-smi unavailable ({e})"
    return q


def run(eng, rec, scale, block, overlap, chunk, ref_blocks):
    import torch
    from oracle import cwt_blocks as B
    from ssqueeze_rs_b200.batch import CwtStream, RecordingFeeder
    N, ch = rec.shape
    cs = CwtStream(eng, ch, N, chunk, block, overlap, fs=30000.0, nv=32)
    ns = cs.ns
    mag = torch.zeros((ch, ns), dtype=torch.float32, device="cuda")
    evs = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with RecordingFeeder(eng, rec, None, chunk=chunk, scale=scale, stream=cs) as feed:
        while True:
            a = torch.cuda.Event(enable_timing=True)
            b = torch.cuda.Event(enable_timing=True)
            a.record()
            Tx = feed.push_next()
            b.record()
            if Tx is None:
                break
            evs.append((a, b))
            if Tx.shape[2]:
                mag += Tx.abs().sum(dim=2)
            del Tx
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    name = eng.last_kernel_name()
    push_ms = sum(a.elapsed_time(b) for a, b in evs)
    cs.close()
    # the batch call on the materialised extended blocks 1 .. ref_blocks (all channels of a block in one call)
    x = torch.from_numpy(np.asarray(rec[: (ref_blocks + 2) * block + overlap]).astype(np.float32) * np.float32(scale))
    ref_ms = 0.0
    for b in range(1, ref_blocks + 1):
        e = torch.from_numpy(np.ascontiguousarray(B.extended_block(x.numpy(), block, overlap, b).T)).cuda()
        sc = cs.scales
        eng.ssq_cwt(e, scales=sc, fs=30000.0)  # warm-up of this shape
        a = torch.cuda.Event(enable_timing=True)
        z = torch.cuda.Event(enable_timing=True)
        a.record()
        out = eng.ssq_cwt(e, scales=sc, fs=30000.0)
        z.record()
        torch.cuda.synchronize()
        ref_ms += a.elapsed_time(z)
        del out
    nblk = B.n_blocks(N, block)
    e_len = block + 2 * overlap
    L = 1 << int(np.ceil(np.log2(e_len + e_len // 2)))
    return dict(block=block, overlap=overlap, ns=ns, L=L, chunk=chunk, kernel=name,
                feeder_msamples_per_s=ch * N / wall / 1e6, feeder_wall_s=wall, pushes=len(evs),
                push_device_ms=push_ms, stream_ms_per_block=push_ms / nblk,
                batch_materialised_ms_per_block=ref_ms / ref_blocks, mag_checksum=float(mag.sum()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--log2n", type=int, default=22)
    ap.add_argument("--geometries", default="17:14,14:12", help="log2 block:log2 overlap, comma separated")
    ap.add_argument("--chunk", type=int, default=1 << 17)
    ap.add_argument("--ref-blocks", type=int, default=4)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch
    from ssqueeze_rs_b200.batch import Engine
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this tool measures the B200 and has no CPU mode")
    eng = Engine(0)
    N = 1 << a.log2n
    res = dict(card=card(), channels=a.channels, samples=N, results=[])
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "rec.dat")
        rng = np.random.default_rng(0)
        mm = np.memmap(path, dtype=np.int16, mode="w+", shape=(N, a.channels))
        step = 1 << 18
        for i in range(0, N, step):
            m = min(step, N - i)
            t = (np.arange(i, i + m) / 30000.0)[:, None]
            mm[i:i + m] = (600 * np.sin(2 * np.pi * (40 + 30 * t) * t) + rng.normal(0, 200, (m, a.channels))).astype(np.int16)
        mm.flush()
        del mm
        rec = np.memmap(path, dtype=np.int16, mode="r").reshape(N, a.channels)
        for g in a.geometries.split(","):
            lb, lo = (int(v) for v in g.split(":"))
            r = run(eng, rec, 0.195, 1 << lb, 1 << lo, a.chunk, a.ref_blocks)
            res["results"].append(r)
            print(json.dumps(r), flush=True)
    print(json.dumps(dict(card=res["card"])))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

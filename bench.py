#!/usr/bin/env python
"""bench.py -- ssq_stft input Msamples/s on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A step = one pass of the fused ssq_stft kernel over one batch of synthetic
multichannel input.  N=1 workload = BASELINE.json configs[1]: 384 channels x
60 s @ 30 kHz (1.8 M samples), n_fft=512, hop=32, Hann window, reflect pad.
N>1: every rank processes its own 384-channel batch (channels are independent
units; no data-path collective) -> weak scaling; value = all ranks' samples /
max-over-ranks device time.

`value`  : inputs already resident in HBM, device time by CUDA events.
`e2e`    : same metric through the C ABI with HOST (pinned) buffers, H2D and
           D2H copies of every byte inside the timed region.
`--impl reference`: the reference's own algorithm on the host cores (the C
           restatement oracle/ssq_stft_ref.c, as-written variant; the Rust
           crate cannot be built in this image), rank 0 only, bounded sample.
`--dump-outputs DIR`: after the timed steps, rank 0 writes a fixed, seeded
           sample of the Tx its last step computed to DIR/Tx.npy (see
           dump_outputs), so that two builds can be compared on the same input.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FS = 30000.0
N_FFT, HOP = 512, 32
CHANNELS = 384
SAMPLES = 1_800_000
WORKLOAD = "ssq_stft 384ch x 1.8M samples (60 s @ 30 kHz) synthetic neural, n_fft=512 hop=32 hann reflect"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel on the default workload, from
    the ncu pass recorded in profiles/bench_dram.json by tools/record_dram.py (which stores the commit it was taken
    at).  (None, why) when the record is missing or was taken on another kernel build."""
    path = os.path.join(ROOT, "profiles", "bench_dram.json")
    try:
        rec = json.load(open(path))
        return float(rec["dram_bytes_per_launch"]), {"file": "profiles/bench_dram.json", "commit": rec.get("commit"),
                                                     "kernel_sources_sha": rec.get("kernel_sources_sha"),
                                                     "current_kernel_sources_sha": kernel_sources_sha()}
    except Exception as e:  # noqa: BLE001
        return None, {"unavailable": str(e)}


def kernel_sources_sha():
    """Fingerprint of the CUDA sources the benchmarked kernel is built from (so a stale ncu record shows)."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "ssqueeze_rs_b200", "csrc")
    for f in ("stft_h32r.cuh", "fft_regs.cuh", "stft_kernels.cuh", "ssq_common.cuh"):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def algorithmic_bytes(channels, n, n_fft=N_FFT, hop=HOP):
    """SURVEY 8(d): B = C*(4*N + 8*n_freqs*n_frames)."""
    n_freqs, n_frames = n_fft // 2 + 1, (n - 1) // hop + 1
    return channels * (4 * n + 8 * n_freqs * n_frames)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [ln for (t, ln) in self.lines if t_begin is None or (t_begin <= t <= t_end + 0.06)]
        if not lines:  # region shorter than one sampling period: nearest samples around it
            lines = [ln for (t, ln) in self.lines if t_begin - 0.3 <= t <= t_end + 0.3]
        for ln in lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_neural(torch, channels, n, fs, device, seed):
    """SURVEY 8(d) 'neural' recipe, generated on the device: 50*pink(0.5-300 Hz) +
    20*sin(2pi 8 t + phi) + 10*sin(2pi (40 + 20 sin 2pi 0.2 t) t) + 5*sin(2pi 60 t) +
    10*N(0,1) + Poisson(20 Hz) biphasic 1.5 ms spikes of 80-200 uV."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    x = torch.empty((channels, n), dtype=torch.float32, device=device)
    t = torch.arange(n, device=device, dtype=torch.float64) / fs
    base = (10.0 * torch.sin(2 * np.pi * (40.0 + 20.0 * torch.sin(2 * np.pi * 0.2 * t)) * t)
            + 5.0 * torch.sin(2 * np.pi * 60.0 * t)).to(torch.float32)
    freqs = torch.fft.rfftfreq(n, d=1.0 / fs).to(device)
    shape = torch.where((freqs >= 0.5) & (freqs <= 300.0), 1.0 / torch.sqrt(torch.clamp(freqs, min=0.5)),
                        torch.zeros_like(freqs)).to(torch.float32)
    L = int(0.0015 * fs)
    tt = torch.arange(L, device=device, dtype=torch.float32) / L
    templ = (torch.sin(2 * np.pi * tt) * torch.hann_window(L, device=device)).view(1, 1, L)
    step = 16
    for c0 in range(0, channels, step):
        c1 = min(channels, c0 + step)
        m = c1 - c0
        white = torch.randn((m, n), generator=g, device=device, dtype=torch.float32)
        pink = torch.fft.irfft(torch.fft.rfft(white) * shape, n=n)
        pink = pink / pink.std(dim=1, keepdim=True).clamp_min(1e-12)
        phi = torch.rand((m, 1), generator=g, device=device, dtype=torch.float64) * 2 * np.pi
        theta = torch.sin(2 * np.pi * 8.0 * t.view(1, -1) + phi).to(torch.float32)
        spikes = (torch.rand((m, n), generator=g, device=device) < (20.0 / fs)).to(torch.float32)
        amp = 80.0 + 120.0 * torch.rand((m, n), generator=g, device=device)
        sp = torch.nn.functional.conv1d((spikes * amp).view(m, 1, n), templ, padding=L // 2)[:, 0, :n]
        x[c0:c1] = (50.0 * pink + 20.0 * theta + base.view(1, -1)
                    + 10.0 * torch.randn((m, n), generator=g, device=device) + sp)
        del white, pink, theta, spikes, amp, sp
    return x


def make_neural_cpu(channels, n, fs, seed):
    """Same recipe on the host (numpy) for the CPU reference arm's bounded sample."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / fs
    out = np.empty((channels, n))
    f = np.fft.rfftfreq(n, 1.0 / fs)
    shape = np.where((f >= 0.5) & (f <= 300.0), 1.0 / np.sqrt(np.maximum(f, 0.5)), 0.0)
    for c in range(channels):
        pink = np.fft.irfft(np.fft.rfft(rng.standard_normal(n)) * shape, n=n)
        pink /= max(pink.std(), 1e-12)
        sp = np.zeros(n)
        idx = np.nonzero(rng.random(n) < 20.0 / fs)[0]
        L = int(0.0015 * fs)
        templ = np.sin(2 * np.pi * np.arange(L) / L) * np.hanning(L)
        for i in idx:
            a = 80 + 120 * rng.random()
            e = min(n, i + L)
            sp[i:e] += a * templ[:e - i]
        out[c] = (50 * pink + 20 * np.sin(2 * np.pi * 8 * t + rng.random() * 2 * np.pi)
                  + 10 * np.sin(2 * np.pi * (40 + 20 * np.sin(2 * np.pi * 0.2 * t)) * t)
                  + 5 * np.sin(2 * np.pi * 60 * t) + 10 * rng.standard_normal(n) + sp)
    return out


DUMP_COLUMNS = 16384  # x 257 bins x 8 bytes = 34 MB: a dump stays under 64 MB
DUMP_SEED = 0x5351


def dump_outputs(path, Tx):
    """Writes a fixed sample of Tx [channels, n_freqs, n_frames] (complex64, on the device) to path/Tx.npy:
    DUMP_COLUMNS (channel, frame) columns drawn without replacement by a generator seeded with DUMP_SEED, in
    ascending (channel, frame) order, as float32 [columns, n_freqs, 2] (real, imaginary).  The columns depend only on
    the shape of Tx, so two runs with the same arguments dump the same columns."""
    import torch
    ch, _, nfr = Tx.shape
    k = min(DUMP_COLUMNS, ch * nfr)
    flat = np.sort(np.random.default_rng(DUMP_SEED).choice(ch * nfr, size=k, replace=False))
    c = torch.from_numpy(flat // nfr).to(Tx.device)
    f = torch.from_numpy(flat % nfr).to(Tx.device)
    cols = torch.view_as_real(Tx[c, :, f]).cpu().numpy()
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "Tx.npy"), cols.astype(np.float32, copy=False))


def cpu_reference_run(n_samples, steps, warmup, mode=0, channels=1):
    """Times the C restatement (oracle/ssq_stft_ref.c) on `channels` x n_samples."""
    from oracle import cref
    cref.use_all_cores()
    x = make_neural_cpu(channels, n_samples, FS, 0x5351)
    w = np.hanning(N_FFT)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for c in range(channels):
            cref.ssq_stft(x[c], w, N_FFT, HOP, FS, mode=mode)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return channels * n_samples / (sum(times) / len(times)) / 1e6, cref.num_threads(), sum(times) / len(times)


def parity_gates(eng, torch, dev, n_samples=200_000):
    """SURVEY 8(d) parity gates, reported beside the throughput: the benchmarked kernel against the float64 oracle
    (the checker, part of the cpu_baseline leg) on one channel of the same synthetic recipe.  The destination bin of
    every (source bin, frame) is written by the kernel itself (diagnostic compile-time variant, asserted bit-equal to
    the timed kernel's Tx); every bin that differs from the reference's arg-min is classified by oracle/parity.py."""
    from oracle import parity as P
    from oracle import ssq_oracle as O
    x = make_neural_cpu(1, n_samples, FS, 0x5351 + 7)
    w = np.hanning(N_FFT)
    ref, _, ao = O.ssq_stft(x[0], w, n_fft=N_FFT, hop_len=HOP, fs=FS, return_aux=True)
    xd = torch.from_numpy(x.astype(np.float32)).to(dev)
    Tx_d, aux = eng.ssq_stft(xd, w, n_fft=N_FFT, hop_len=HOP, fs=FS, return_aux=True)
    kernel = eng.last_kernel_name()
    Tx_p = eng.ssq_stft(xd, w, n_fft=N_FFT, hop_len=HOP, fs=FS)
    torch.cuda.synchronize()
    same = bool(torch.equal(Tx_d, Tx_p))
    got = Tx_p[0].cpu().numpy().astype(np.complex128)
    kb = aux["kb"][0].cpu().numpy()
    rep = P.public(P.classify_stft_bins(kb, ao, N_FFT, FS, None, w_dev=aux["w"][0].cpu().numpy().astype(np.float64)))
    scale = float(np.abs(ref).max())
    Tacc = P.reaccumulate(ao["Sx"], kb, FS)
    good = ~(kb != ao["k"]).any(axis=0)
    cs = np.abs(got.sum(axis=0) - ref.sum(axis=0)).max() / np.abs(ref.sum(axis=0)).max()
    rep.update({
        "against": "oracle/ssq_oracle.py (f64), 1 channel x %d samples of the bench recipe" % n_samples,
        "kernel": kernel, "diagnostic_variant_bit_equal_to_timed_kernel": same,
        "Sx_rel_max_err": float(np.abs(aux["Sx"][0].cpu().numpy() - ao["Sx"]).max() / np.abs(ao["Sx"]).max()),
        "Tx_rel_max_err_vs_reference_accumulation_over_device_bins": float(np.abs(got - Tacc).max() / scale),
        "Tx_rel_max_err_on_columns_without_flip": float(np.abs(got[:, good] - ref[:, good]).max() / scale) if good.any() else None,
        "columns_without_flip": int(good.sum()), "columns_total": int(good.size),
        "column_sum_rel_err": float(cs), "rtol": 1e-4})
    return rep


# ---------------------------------------------------------------------------------------------------------
# The other named configs of BASELINE.json, as sub-records of the same JSON line (`configs`): device-timed,
# channels sharded over the ranks (strong scaling), each with its own roofline, a parity check of the CUDA path
# against the oracle on a cut, and a CPU baseline (rank 0 of a 1-GPU run only).
# ---------------------------------------------------------------------------------------------------------
def _timed(torch, stream, step, warmup, steps, dev):
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(steps):
            step()
        ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps


def _record(name, units_rank, ms_rank, abytes_rank, dev, world, desc, kernel, extra):
    """Per-rank figures of one side config; side_configs() turns them into the job's record (collectives there, so
    that a rank that failed cannot leave the others waiting inside an all-reduce)."""
    return dict(name=name, units=units_rank, ms=ms_rank, abytes=abytes_rank, desc=desc, kernel=kernel, extra=extra)


def _finish_record(r, dev, world):
    from ssqueeze_rs_b200.dist import job_throughput, sum_over_ranks
    name, units_rank, ms_rank, abytes_rank, desc, kernel, extra = (r[k] for k in ("name", "units", "ms", "abytes", "desc", "kernel", "extra"))
    per_s, ms = job_throughput(units_rank, ms_rank, dev)
    ab = sum_over_ranks(abytes_rank, dev)
    peak, peak_src = measured_peak_gbs()
    ach = ab / (ms * 1e-3) / 1e9 / world  # per GPU
    rec = {"metric": f"{name} input Msamples/s", "value": per_s / 1e6, "unit": "Msamples/s", "ms_per_step": ms,
           "scaling": "strong", "config": {"workload": desc},
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                        "peak_source": peak_src, "algorithmic_bytes_per_step": ab,
                        "note": "per GPU; whole step (all kernels of the call), not one kernel"},
           "kernel": kernel}
    rec.update(extra)
    if rec.get("scaling") == "weak":
        rec["roofline"]["note"] = "per GPU; wall clock of the whole host-to-host step"
    return rec


def side_c5(torch, eng, dev, rank, world, stream, g, cpu, scale=1.0):
    """BASELINE configs[4]: 1024 channels x 10 min @ 30 kHz (18 M samples), 1024 / world channels per GPU, input
    resident (73.7 GB at world 1), Tx through a ring of two 16-channel output buffers as a host gather would drain
    them.  Input: white noise + two tones (the neural recipe needs an 18 M-point FFT per channel block to generate)."""
    from oracle import parity as P
    from oracle import ssq_oracle as O
    ch_total, n = max(world, int(1024 * scale)), int(18_000_000 * (scale if scale < 1 else 1))
    c0, c1 = ch_total * rank // world, ch_total * (rank + 1) // world
    ch, blk = c1 - c0, 16
    win = np.hanning(N_FFT)
    x = torch.empty((ch, n), dtype=torch.float32, device=dev)
    tt = torch.arange(n, device=dev, dtype=torch.float32) / FS
    tone = 20.0 * torch.sin(2 * np.pi * 8.0 * tt) + 5.0 * torch.sin(2 * np.pi * 60.0 * tt)
    for b0 in range(0, ch, blk):
        x[b0:b0 + blk] = torch.randn((min(blk, ch - b0), n), generator=g, device=dev) * 10 + tone
    del tt, tone
    nfr = (n - 1) // HOP + 1
    ring = [torch.empty((blk, N_FFT // 2 + 1, nfr), dtype=torch.complex64, device=dev) for _ in range(2)]

    def step():
        for i, b0 in enumerate(range(0, ch, blk)):
            m = min(blk, ch - b0)
            eng.ssq_stft(x[b0:b0 + m], win, N_FFT, HOP, FS, out=ring[i & 1][:m])

    ms = _timed(torch, stream, step, 1, 2, dev)
    extra = {}
    if rank == 0:
        # parity: slices of frames at the start, far into and at the end of the recording (a frame depends on its own
        # 512 samples only), every bin classified
        tot = dict(bins_total=0, mismatch_total=0, within_edge=0, ill_conditioned=0, below_energy_gate=0, unexplained=0,
                   max_err_over_tol=0.0)
        left = (N_FFT - 1) // 2
        for f0, nf in ((0, 64), (nfr // 2, 64), (nfr - 64, 64)):
            g0 = max(0, (f0 * HOP - left) // HOP)
            a, b = g0 * HOP, min(n, (f0 + nf - 1) * HOP - left + N_FFT)
            xs = x[0:1, a:b].contiguous()
            Tx, aux = eng.ssq_stft(xs, win, N_FFT, HOP, FS, return_aux=True)
            _, _, ao = O.ssq_stft(xs[0].cpu().numpy().astype(np.float64), win, n_fft=N_FFT, hop_len=HOP, fs=FS, return_aux=True)
            r = P.classify_stft_bins(aux["kb"][0].cpu().numpy(), ao, N_FFT, FS, None, w_dev=aux["w"][0].cpu().numpy().astype(np.float64))
            for k in tot:
                tot[k] = max(tot[k], r[k]) if k == "max_err_over_tol" else tot[k] + r[k]
        tot["against"] = "oracle/ssq_oracle.py on three 64-frame slices of channel 0 (start, middle, end)"
        extra["parity"] = tot
        if cpu:
            msps, threads, sec = cpu_reference_run(450_000, 1, 0, mode=0)
            extra["cpu_baseline"] = {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": "port",
                                     "sample": f"1 channel x 450000 samples ({sec:.1f} s), C restatement of ssq_stft.rs as written"}
    rec = _record("ssq_stft(c5)", float(ch) * n, ms, algorithmic_bytes(ch, n), dev, world,
                  f"ssq_stft configs[4]: {ch_total}ch x {n} samples over {world} GPU(s), blocks of {blk} channels through a "
                  f"ring of 2 output buffers, n_fft=512 hop=32; white noise + tones", eng.last_kernel_name(), extra)
    del x, ring
    torch.cuda.empty_cache()
    return rec


def side_c4_istft(torch, eng, dev, rank, world, stream, g, cpu, scale=1.0):
    """BASELINE configs[3]: istft on 4096 channels x 10 s @ 30 kHz (300 k samples), n_fft=512 hop=32 (overlap-add +
    window norm + unpad); Sx produced on the device by the stft kernel (78.9 GB at world 1)."""
    from oracle import ssq_oracle as O
    ch_total, n = max(world, int(4096 * scale)), 300_000
    c0, c1 = ch_total * rank // world, ch_total * (rank + 1) // world
    ch = c1 - c0
    win = np.hanning(N_FFT)
    x = torch.randn((ch, n), generator=g, device=dev) * 10
    nfr = (n - 1) // HOP + 1
    Sx = torch.empty((ch, N_FFT // 2 + 1, nfr), dtype=torch.complex64, device=dev)
    for b0 in range(0, ch, 256):
        eng.stft(x[b0:b0 + 256], win, N_FFT, HOP, out=Sx[b0:b0 + 256])
    out = {"x": torch.empty((ch, n), dtype=torch.float32, device=dev)}

    def step():
        eng.istft(Sx, win, N_FFT, HOP, N=n, out=out["x"])

    ms = _timed(torch, stream, step, 2, 3, dev)
    extra = {}
    if rank == 0:
        xr = out["x"]
        mae = float((xr - x).abs().mean())
        So = Sx[0].cpu().numpy().astype(np.complex128)
        xo = O.istft(So, win, n_fft=N_FFT, hop_len=HOP, N=n)
        err = float(np.abs(xr[0].cpu().numpy() - xo).max() / np.abs(xo).max())
        extra["parity"] = {"against": "oracle/ssq_oracle.py istft on channel 0 (same Sx)", "rel_max_err": err, "rtol": 1e-4,
                           "within_rtol": bool(err < 1e-4), "round_trip_mae_all_channels": mae,
                           "round_trip_mae_rel": mae / float(x.abs().mean())}
        if cpu:
            t0 = time.perf_counter()
            O.istft(So, win, n_fft=N_FFT, hop_len=HOP, N=n)
            sec = time.perf_counter() - t0
            extra["cpu_baseline"] = {"value": n / sec / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
                                     "sample": f"1 channel x {n} samples ({sec:.2f} s), NumPy oracle (pocketfft irfft + overlap-add loop); "
                                               "the reference crate has no istft"}
    rec = _record("istft", float(ch) * n, ms, ch * (4 * n + 8 * (N_FFT // 2 + 1) * nfr), dev, world,
                  f"istft configs[3]: {ch_total}ch x {n} samples over {world} GPU(s), n_fft=512 hop=32", eng.last_kernel_name(), extra)
    del x, Sx, out
    torch.cuda.empty_cache()
    return rec


def side_c3_ssq_cwt(torch, eng, dev, rank, world, stream, g, cpu, scale=1.0):
    """BASELINE configs[2]: ssq_cwt GMW nv=32 (576 scales) on 64 channels x 2^20 chirp+noise; Tx (4.8 GB per channel)
    through a ring of two 4-channel output buffers."""
    from oracle import parity as P
    from oracle import ssq_oracle as O
    ch_total, n = max(world, int(64 * scale)), 1 << 20
    c0, c1 = ch_total * rank // world, ch_total * (rank + 1) // world
    ch, blk = c1 - c0, 4
    t = torch.arange(n, device=dev, dtype=torch.float64) / n
    chirp = torch.sin(2 * np.pi * n * (0.001 * t + 0.5 * 0.399 * t * t)).to(torch.float32)
    x = chirp.view(1, -1) + 0.5 * torch.randn((ch, n), generator=g, device=dev)
    sc = eng.default_scales(n, 32)
    ns = len(sc)
    ring = [torch.empty((blk, ns, n), dtype=torch.complex64, device=dev) for _ in range(2)]

    def step():
        for i, b0 in enumerate(range(0, ch, blk)):
            m = min(blk, ch - b0)
            eng.ssq_cwt(x[b0:b0 + m], "gmw", sc, fs=1.0, nv=32, maprange="maximal", out=ring[i & 1][:m])

    ms = _timed(torch, stream, step, 1, 2, dev)
    kernel = eng.last_kernel_name()
    extra = {}
    del ring
    torch.cuda.empty_cache()
    if rank == 0:
        # parity on a 2^16-sample cut of channel 0 (the float64 oracle needs 2 x ns x pad_len complex128: 80 GB at 2^20)
        m = 1 << 17
        xs = x[0:1, :m].contiguous()
        Tx, sf, aux = eng.ssq_cwt(xs, "gmw", None, fs=1.0, nv=32, maprange="maximal", return_aux=True)
        xs64 = xs[0].cpu().numpy().astype(np.float64)
        t0 = time.perf_counter()
        To, sfo, ao = O.ssq_cwt(xs64, "gmw", None, fs=1.0, nv=32, maprange="maximal", return_aux=True)
        sec = time.perf_counter() - t0
        kb = aux["kb"][0].cpu().numpy()
        r = P.public(P.classify_cwt_bins(kb, ao, xs64, "gmw", 1.0, "reflect", sfo, w_dev=aux["w"][0].cpu().numpy().astype(np.float64)))
        Tacc = P.reaccumulate_cwt(ao["Wx"], kb, To.shape[0])
        r["Tx_rel_max_err_vs_reference_accumulation_over_device_rows"] = float(
            np.abs(Tx[0].cpu().numpy().astype(np.complex128) - Tacc).max() / np.abs(To).max())
        r["against"] = f"oracle/ssq_oracle.py ssq_cwt (f64) on a {m}-sample cut of channel 0, nv=32 ({To.shape[0]} scales)"
        r["kernel"] = eng.last_kernel_name()
        extra["parity"] = r
        if cpu:
            extra["cpu_baseline"] = {"value": m / sec / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
                                     "sample": f"1 channel x {m} samples, {To.shape[0]} scales ({sec:.1f} s), NumPy oracle restating "
                                               "ssq_cwt.rs (pocketfft); the full-size case needs > 80 GB in float64 (SURVEY 8a row 15)"}
    rec = _record("ssq_cwt", float(ch) * n, ms, ch * (4 * n + 8 * ns * n), dev, world,
                  f"ssq_cwt configs[2]: gmw nv=32 ({ns} scales), {ch_total}ch x {n} chirp+noise over {world} GPU(s), blocks of "
                  f"{blk} channels through a ring of 2 output buffers", kernel, extra)
    del x
    torch.cuda.empty_cache()
    return rec


def side_ridges_e2e(torch, eng, dev, rank, world, stream, g, cpu, scale=1.0):
    """The consumer that stays on the device (SURVEY 8f rank 4): pinned host x -> H2D -> ssq_stft (configs[1] geometry)
    -> ridge extraction on Tx where it lies in HBM -> D2H of the ridge indices only (0.2 % of Tx's bytes).  Timed end
    to end like `e2e` (host buffers, copies inside the timed region); every rank runs its own batch (weak scaling)."""
    ch, n = max(1, int(CHANNELS * scale)), SAMPLES
    win = np.hanning(N_FFT)
    nfq, nfr = N_FFT // 2 + 1, (n - 1) // HOP + 1
    xh = torch.empty((ch, n), dtype=torch.float32, pin_memory=True)
    xh.copy_(make_neural(torch, ch, n, FS, dev, 0x5351 + rank))
    rh = torch.empty((ch, nfr, 1), dtype=torch.int32, pin_memory=True)
    xd = torch.empty((ch, n), dtype=torch.float32, device=dev)
    Tx = torch.empty((ch, nfq, nfr), dtype=torch.complex64, device=dev)
    sf = np.arange(nfq) * 0.5 / (nfq - 1) + 1e-9  # normalised frequencies (upstream's `scales` for an STFT map)
    torch.cuda.synchronize()

    def step():
        with torch.cuda.stream(stream):
            xd.copy_(xh, non_blocking=True)
            eng.ssq_stft(xd, win, N_FFT, HOP, FS, out=Tx, modulated=True)
            idx = eng.extract_ridges(Tx, sf, penalty=2.0, n_ridges=1, bw=4, transform="stft")
            rh.copy_(idx, non_blocking=True)
        stream.synchronize()

    step()
    t0 = time.perf_counter()
    steps = 2
    for _ in range(steps):
        step()
    ms = (time.perf_counter() - t0) / steps * 1e3
    med = float(np.median(rh[0, :, 0].numpy()))
    rec = _record("ssq_stft+extract_ridges (e2e)", float(ch) * n, ms, algorithmic_bytes(ch, n), dev, world,
                  f"configs[1] geometry, {ch}ch x {n} per GPU: host x -> ssq_stft(modulated) -> extract_ridges(penalty 2, 1 ridge) "
                  f"on device -> host ridge indices", "ssq_stft512_h32r_kernel<ssq> + ridge_forward_kernel",
                  {"e2e": {"h2d_bytes_per_step": int(ch * n * 4), "d2h_bytes_per_step": int(ch * nfr * 4),
                           "note": "wall clock around the public Engine calls, pinned host in/out"},
                   "scaling": "weak", "median_ridge_bin_channel0": med})
    del xd, Tx, xh, rh
    torch.cuda.empty_cache()
    return rec


def side_feeder_e2e(torch, eng, dev, rank, world, stream, g, cpu, scale=1.0):
    """The reader half of the streaming path (SURVEY 8f rank 1): an interleaved int16 (samples, channels) recording in
    PAGEABLE host memory -- what a memory-mapped probe file is -- walked in chunks by RecordingFeeder (ring of pinned
    staging buffers inside the library: host copy | H2D | transform overlap), Tx consumed on the device (band power
    per channel and bin, a reduction) so that only [channels, 257] floats leave it.  Wall clock, host to host."""
    from ssqueeze_rs_b200.batch import RecordingFeeder
    ch, n = max(1, int(CHANNELS * scale)), SAMPLES
    win = np.hanning(N_FFT)
    nfq = N_FFT // 2 + 1
    x = make_neural(torch, ch, n, FS, dev, 0x5351 + rank)
    rec = (x / 0.195).clamp_(-32768, 32767).to(torch.int16).t().contiguous().cpu().numpy()  # pageable [n, ch]
    del x
    torch.cuda.empty_cache()
    ph = torch.empty((ch, nfq), dtype=torch.float32, pin_memory=True)
    chunk = 1 << 15
    split = {}

    def step():
        power = torch.zeros((ch, nfq), dtype=torch.float32, device=dev)
        with torch.cuda.stream(stream):
            ta = time.perf_counter()
            feed = RecordingFeeder(eng, rec, win, N_FFT, HOP, FS, chunk=chunk, scale=0.195, depth=3)
            tb = time.perf_counter()
            for Tx in feed:
                power += torch.view_as_real(Tx).square_().sum(dim=(2, 3))
            ph.copy_(power, non_blocking=True)
            stream.synchronize()
            tc = time.perf_counter()
            feed.close()
            split.update(setup_ms=(tb - ta) * 1e3, stream_ms=(tc - tb) * 1e3, teardown_ms=(time.perf_counter() - tc) * 1e3)

    step()
    t0 = time.perf_counter()
    steps = 2
    for _ in range(steps):
        step()
    ms = (time.perf_counter() - t0) / steps * 1e3
    r = _record("ssq_stft via RecordingFeeder (e2e, int16 host recording)", float(ch) * n, ms, algorithmic_bytes(ch, n),
                dev, world,
                f"configs[1] geometry, {ch}ch x {n} int16 interleaved in pageable host memory, chunks of {chunk} samples "
                f"through ssq_feeder_push (3 pinned slots; stream and feeder created and destroyed inside the timed step), Tx reduced on device to band power [channels, 257]",
                "ssq_stft512_h32r_kernel<ssq> + deinterleave_kernel (+ torch reduction as the consumer)",
                {"e2e": {"h2d_bytes_per_step": int(ch * n * 2), "d2h_bytes_per_step": int(ch * nfq * 4),
                         "note": "wall clock around RecordingFeeder, pageable host in, pinned host out"},
                 "scaling": "weak", "band_power_checksum": float(ph.sum()),
                 "split_ms": {k: round(v, 2) for k, v in split.items()}})
    del rec
    torch.cuda.empty_cache()
    return r


def side_configs(torch, eng, dev, rank, world, stream, cpu, scale=1.0, only=None):
    g = torch.Generator(device=dev)
    g.manual_seed(0x5351 + rank)
    out = {}
    from ssqueeze_rs_b200.dist import max_over_ranks
    for key, fn in (("c5", side_c5), ("c4_istft", side_c4_istft), ("c3_ssq_cwt", side_c3_ssq_cwt),
                    ("c2_ridges_e2e", side_ridges_e2e), ("c2_feeder_e2e", side_feeder_e2e)):
        if only and key not in only:
            continue
        r, err = None, None
        try:
            r = fn(torch, eng, dev, rank, world, stream, g, cpu, scale)
        except Exception as e:  # noqa: BLE001 -- a side record must not take the contract line down with it
            torch.cuda.empty_cache()
            err = f"{type(e).__name__}: {e}"
        failed = max_over_ranks(0.0 if err is None else 1.0, dev)  # every rank takes part, whatever happened to it
        if failed:
            out[key] = {"error": err or "another rank failed"}
        else:
            out[key] = _finish_record(r, dev, world)
    return out



def run_reference(args, rank, world):
    if rank != 0:
        return
    n_s = args.ref_samples
    steps = args.steps
    warm = max(1, min(args.warmup, 3))
    msps, threads, sec = cpu_reference_run(n_s, steps, warm, mode=0)
    line = {
        "impl": "reference", "metric": "ssq_stft input Msamples/s", "value": msps, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_fft": N_FFT, "hop": HOP, "fs": FS},
        "cpu_baseline": {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": "port",
                         "sample": f"1 channel x {n_s} samples per step of the same synthetic recipe; C restatement "
                                   "of ssq_stft.rs as written (frames parallel with a plan per frame, serial phase, "
                                   "serial O(n_freqs^2) arg-min reassignment); OpenMP threads = host cores"},
        "e2e": {"value": msps, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from ssqueeze_rs_b200 import _lib
    from ssqueeze_rs_b200.batch import Engine

    channels, n = args.channels, args.samples
    n_freqs, n_frames = N_FFT // 2 + 1, (n - 1) // HOP + 1
    eng = Engine(local_rank)
    window = np.hanning(N_FFT)
    x = make_neural(torch, channels, n, FS, dev, 0x5351 + rank)
    Tx = torch.empty((channels, n_freqs, n_frames), dtype=torch.complex64, device=dev)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)  # the kernels, the step events and the timed region share this stream
    eng.ctx.set_stream(stream.cuda_stream)

    def step():
        eng.ssq_stft_ptr(x.data_ptr(), channels, n, window, N_FFT, HOP, FS, Tx.data_ptr())

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_begin = time.time()
    launches0 = eng.ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for a, b in kev:
            a.record(stream)
            step()
            b.record(stream)
        ev1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_end = time.time()
    kernel_ms = [a.elapsed_time(b) for a, b in kev]
    clocks = sampler.stop(t_begin, t_end)
    launches = eng.ctx.launch_count() - launches0
    from ssqueeze_rs_b200.dist import job_throughput
    per_s, total_ms = job_throughput(float(channels) * n * args.steps, ev0.elapsed_time(ev1), dev)
    ms_per_step = total_ms / args.steps
    value = per_s / 1e6

    # checksum so the timed work cannot be optimised away / silently skipped
    chk = float(torch.view_as_real(Tx[0, :, :64]).abs().sum().item())
    if not np.isfinite(chk) or chk == 0.0:
        raise SystemExit("bench.py: kernel produced no output")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, Tx)

    # ---- roofline of the dominant kernel (live CUDA-event durations) -----------
    peak, peak_src = measured_peak_gbs()
    kms = float(np.mean(kernel_ms))
    abytes = algorithmic_bytes(channels, n)
    achieved = abytes / (kms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic() if (channels, n) == (CHANNELS, SAMPLES) else (None, {"unavailable": "not the default workload"})
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel_ms": kms, "algorithmic_bytes_per_launch": abytes,
                "peak_source": peak_src, "kernel": eng.last_kernel_name()}
    if (N_FFT, HOP) == (512, 32):
        # what actually binds this kernel (DESIGN 3.1): the on-chip pipes, per frame and SM.  Instruction and wavefront
        # counts are those of the ncu capture profiles/r2/r2m_* of this kernel (979 warp-instructions -- 249 packed
        # fp32x2, which hold the fp32 pipe two cycles, and 97 scalar fp32 among them -- and 341 shared-memory
        # wavefronts per frame); the measured figure comes from this run's kernel time and the clock sampled under load.
        frames = channels * ((n - 1) // HOP + 1)
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        clk = kms * 1e-3 * mhz * 1e6 * sms / frames
        roofline["on_chip"] = {
            "clk_per_frame_per_sm": clk,
            "floors_clk": {"fp32_pipe": (249 * 2 + 97) / 4.0, "issue_slots": 979 / 4.0, "l1tex_wavefronts": 341.0},
            "frac_of_binding_floor": 341.0 / clk,
            "hbm_equivalent_of_fp32_floor_frac": (abytes / (((249 * 2 + 97) / 4.0) * frames / (mhz * 1e6 * sms)) / 1e9) / peak,
            "source": "profiles/r2/r2m_ssq_stft512_h32r_full.csv (ncu --set full of this kernel)"}

    # ---- e2e through the host-buffer C-ABI call --------------------------------
    del Tx
    torch.cuda.empty_cache()
    e2e = run_e2e(eng, args, rank, world, window, x, dev)

    cpu_baseline = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        parity = parity_gates(eng, torch, dev)
        msps, threads, sec = cpu_reference_run(900_000, 1, 0, mode=0)
        msps_i, _, sec_i = cpu_reference_run(900_000, 1, 1, mode=1, channels=2)
        cpu_baseline = {"value": msps, "unit": "Msamples/s", "cores": threads, "kind": "port",
                        "sample": f"1 channel x 900000 samples ({sec:.1f} s), C restatement of ssq_stft.rs as written",
                        "as_intended_value": msps_i,
                        "as_intended_note": "same numerics, shared FFT plan, O(1) binning, parallel phase/reassign; "
                                            f"2 channels x 900000 samples ({sec_i:.1f} s)"}

    configs = None
    if not args.no_side_configs:
        del x
        torch.cuda.empty_cache()
        configs = side_configs(torch, eng, dev, rank, world, stream, cpu=(world == 1 and not args.no_cpu_baseline),
                               scale=args.side_scale, only=[k for k in args.only_side.split(",") if k] or None)

    if rank == 0:
        line = {
            "metric": "ssq_stft input Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "channels_per_gpu": channels, "samples_per_channel": n, "n_fft": N_FFT,
                       "hop": HOP, "fs": FS, "parallelism": f"channel-shard x{world}, no collective",
                       "l2_policy": "inputs (2.8 GB) and outputs (44 GB) per step exceed the 126 MB L2; no flush"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity": parity, "checksum": chk, "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_other(args, rank, world, local_rank):
    """Device-resident timing of the other rows of SURVEY 8 (not the contract line)."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from ssqueeze_rs_b200.batch import Engine
    from ssqueeze_rs_b200.dist import job_throughput
    eng = Engine(local_rank)
    stream = torch.cuda.Stream(device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(0x5351 + rank)
    win = np.hanning(N_FFT)
    wl = args.workload
    if wl == "istft":
        ch, n = (4096, 300_000) if args.channels == CHANNELS else (args.channels, args.samples)
        x = torch.randn((ch, n), generator=g, device=dev) * 10
        Sx = eng.stft(x, win, N_FFT, HOP)
        nfr = Sx.shape[2]
        abytes = ch * (4 * n + 8 * (N_FFT // 2 + 1) * nfr)
        desc = f"istft {ch}ch x {n} samples, n_fft=512 hop=32 (overlap-add + window norm + unpad)"
        step = lambda: eng.istft(Sx, win, N_FFT, HOP, N=n)
    elif wl in ("stft", "ssq_stft"):
        # the same 384 x 1.8 M recording at another geometry (--n-fft / --hop), e.g. the reference's
        # multichannel script (n_fft 1024, hop 256) or its README (256 / 64)
        ch, n = args.channels, args.samples
        nfft, hop = args.n_fft, args.hop
        win = np.hanning(nfft)
        x = make_neural(torch, ch, n, FS, dev, 0x5351 + rank)
        out = torch.empty((ch, nfft // 2 + 1, (n - 1) // hop + 1), dtype=torch.complex64, device=dev)
        abytes = algorithmic_bytes(ch, n, nfft, hop)
        desc = f"{wl} {ch}ch x {n} samples, n_fft={nfft} hop={hop}"
        if wl == "stft":
            step = lambda: eng.stft(x, win, nfft, hop, out=out)
        else:
            step = lambda: eng.ssq_stft(x, win, nfft, hop, FS, out=out)
    elif wl == "c5":
        # BASELINE configs[4]: 1024 channels x 10 min @ 30 kHz (18 M samples), strong scaling: 1024 / world channels
        # per GPU, resident input (73.7 GB at world 1), Tx written through a ring of two 16-channel buffers
        # (18.5 GB each) as the host gather would drain them.  Input: white noise + two tones (the neural recipe
        # needs an 18 M-point FFT per channel block to generate).
        ch_total, n = (1024, 18_000_000) if args.channels == CHANNELS else (args.channels, args.samples)
        ch = ch_total // world
        blk = 16
        x = torch.empty((ch, n), dtype=torch.float32, device=dev)
        tt = torch.arange(n, device=dev, dtype=torch.float32) / FS
        tone = 20.0 * torch.sin(2 * np.pi * 8.0 * tt) + 5.0 * torch.sin(2 * np.pi * 60.0 * tt)
        for c0 in range(0, ch, blk):
            x[c0:c0 + blk] = torch.randn((min(blk, ch - c0), n), generator=g, device=dev) * 10 + tone
        del tt, tone
        nfr = (n - 1) // HOP + 1
        ring = [torch.empty((blk, N_FFT // 2 + 1, nfr), dtype=torch.complex64, device=dev) for _ in range(2)]
        abytes = algorithmic_bytes(ch, n)
        desc = (f"ssq_stft configs[4]: {ch_total}ch x {n} samples over {world} GPU(s), {ch} ch per GPU in blocks of "
                f"{blk} through a ring of 2 output buffers, n_fft=512 hop=32; white noise + tones")

        def step():
            for i, c0 in enumerate(range(0, ch, blk)):
                m = min(blk, ch - c0)
                eng.ssq_stft(x[c0:c0 + m], win, N_FFT, HOP, FS, out=ring[i & 1][:m])
    else:
        ch, n = (8, 1 << 20) if args.channels == CHANNELS else (args.channels, args.samples)
        t = torch.arange(n, device=dev, dtype=torch.float64) / n
        chirp = torch.sin(2 * np.pi * n * (0.001 * t + 0.5 * 0.399 * t * t)).to(torch.float32)
        x = chirp.view(1, -1) + 0.5 * torch.randn((ch, n), generator=g, device=dev)
        import ctypes as C
        from ssqueeze_rs_b200._lib import load
        ns = load().ssq_cwt_default_scales(n, 32, 0, C.c_void_p(0))
        out = torch.empty((ch, ns, n), dtype=torch.complex64, device=dev)
        abytes = ch * (4 * n + 8 * ns * n)
        desc = f"ssq_cwt gmw nv=32 ({ns} scales) on {ch}ch x {n} chirp+noise (channel cut of configs[2])"
        step = lambda: eng.ssq_cwt(x, "gmw", None, fs=1.0, nv=32, maprange="maximal", out=out)
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        ev1.record(stream)
    torch.cuda.synchronize()
    per_s, total_ms = job_throughput(float(ch) * n * args.steps, ev0.elapsed_time(ev1), dev)
    peak, peak_src = measured_peak_gbs()
    ms = total_ms / args.steps
    if rank == 0:
        print(json.dumps({
            "metric": f"{wl} input Msamples/s", "value": per_s / 1e6, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if wl == "c5" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": desc},
            "roofline": {"bound": "hbm", "achieved": abytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": abytes / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "note": "whole step (all kernels of the call), not one kernel"},
            "kernel": eng.last_kernel_name()}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _pinned_near(nbytes, device):
    """Pinned host bytes on the GPU's NUMA node (ssq_host_alloc_near); returns (numpy uint8 view, address)."""
    import ctypes as C
    from ssqueeze_rs_b200._lib import load
    p = C.c_void_p()
    if load().ssq_host_alloc_near(C.byref(p), nbytes, device) != 0 or not p.value:
        return None, None
    return np.frombuffer((C.c_char * nbytes).from_address(p.value), dtype=np.uint8), p


def run_e2e(eng, args, rank, world, window, x_dev, dev):
    """Host pinned x -> [H2D, kernel, D2H] -> host pinned Tx, every step; then the box's own ceiling for the
    dominant transfer (plain D2H copies of the same size into the same buffers, all ranks at once)."""
    import torch
    import torch.distributed as dist
    import psutil
    from ssqueeze_rs_b200._lib import load
    n = args.samples
    n_freqs, n_frames = N_FFT // 2 + 1, (n - 1) // HOP + 1
    per_ch = n * 4 + n_freqs * n_frames * 8
    avail = psutil.virtual_memory().available
    ch = int(min(args.channels, max(1, (0.45 * avail / max(1, world)) // per_ch)))
    if args.e2e_channels:
        ch = min(ch, args.e2e_channels)
    xb = tb = None
    while ch >= 1:
        xb, xp = _pinned_near(ch * n * 4, dev.index)
        tb, tp = _pinned_near(ch * n_freqs * n_frames * 8, dev.index) if xb is not None else (None, None)
        if tb is not None:
            break
        if xb is not None:
            load().ssq_host_free(xp)
        xb = tb = None
        ch //= 2
    if tb is None:
        return {"value": None, "unit": "Msamples/s", "note": "could not pin host memory"}
    xh = torch.from_numpy(xb.view(np.float32).reshape(ch, n))
    th = tb.view(np.complex64).reshape(ch, n_freqs, n_frames)
    xh.copy_(x_dev[:ch])
    torch.cuda.synchronize()
    steps = max(1, min(args.steps, 3))

    def step():
        eng.ssq_stft_host(xp.value, ch, n, window, N_FFT, HOP, FS, tp.value)

    step()  # warm-up (allocates the device ring)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    val = world * ch * n / (dt / steps) / 1e6
    chk = float(np.abs(th[0, :, :64]).sum())
    d2h = ch * n_freqs * n_frames * 8
    # ---- the ceiling: nothing but D2H copies into the same pinned buffer, every rank at the same time ----
    scratch = torch.empty(min(d2h, 4 << 30), dtype=torch.uint8, device=dev)
    cs = torch.cuda.Stream(dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0 = time.perf_counter()
    off = 0
    while off < d2h:
        m = min(scratch.numel(), d2h - off)
        if load().ssq_memcpy_async(tp.value + off, scratch.data_ptr(), m, 2, cs.cuda_stream) != 0:
            raise SystemExit("bench.py: ssq_memcpy_async failed")
        off += m
    cs.synchronize()
    cdt = torch.tensor([time.perf_counter() - c0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(cdt, op=dist.ReduceOp.MAX)
    ceiling = world * d2h / float(cdt.item()) / 1e9
    achieved = world * d2h / (dt / steps) / 1e9
    node = __import__("ctypes").c_int(-2)
    load().ssq_device_numa_node(dev.index, __import__("ctypes").byref(node))
    del scratch
    load().ssq_host_free(xp)
    load().ssq_host_free(tp)
    return {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": int(ch * n * 4),
            "d2h_bytes_per_step": int(d2h), "channels_per_gpu": ch, "steps": steps,
            "ms_per_step": dt / steps * 1e3, "checksum": chk,
            "d2h_gbs_achieved": achieved, "host_ceiling_gbs": ceiling, "frac_of_host_ceiling": achieved / ceiling,
            "host_ceiling_note": "aggregate GB/s of plain cudaMemcpyAsync D2H copies of the same bytes into the same pinned "
                                 "buffers, all ranks at once (no kernel, no H2D)",
            "pinned_alloc": f"ssq_host_alloc_near (NUMA node of this rank's GPU: {node.value})",
            "note": "ssq_ssq_stft_host_f32: pinned host in/out, chunked H2D|kernel|D2H pipeline inside the call"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--channels", type=int, default=CHANNELS)
    ap.add_argument("--samples", type=int, default=SAMPLES)
    ap.add_argument("--e2e-channels", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the c5 / c4_istft / c3_ssq_cwt sub-records")
    ap.add_argument("--only-side", default="", help="comma-separated keys of the side records to run (default: all)")
    ap.add_argument("--side-scale", type=float, default=1.0, help="shrink the side configs (channels, c5 length) for smoke runs")
    ap.add_argument("--ref-samples", type=int, default=450_000, help="samples per step of the reference arm")
    ap.add_argument("--n-fft", type=int, default=N_FFT, help="side workloads only: another STFT geometry")
    ap.add_argument("--hop", type=int, default=HOP)
    ap.add_argument("--workload", default="ssq_stft", choices=["ssq_stft", "stft", "istft", "ssq_cwt", "c5"],
                    help="ssq_stft (default, BASELINE configs[1]) is the contract line; the others time the "
                         "remaining rows of SURVEY 8 (configs[3] istft 4096 ch x 300 k, configs[2] ssq_cwt on a "
                         "channel cut of 2^20 samples, stft on configs[1]) with the same JSON layout")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="default workload only: write a seeded sample of the last timed step's Tx to DIR/Tx.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    other = args.workload != "ssq_stft" or (args.n_fft, args.hop) != (N_FFT, HOP)
    if args.dump_outputs and (args.impl == "reference" or other):
        ap.error("--dump-outputs is supported for the default workload (ssq_stft, n_fft 512, hop 32) only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif other:
        run_other(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

"""Throughput of the BS.1770-4 loudness path (omega4_b200.loudness) on one GPU, with an oracle check.

    python tools/loudness_bench.py [--warmup 3] [--steps 10] [--out profiles/r03_loudness_bench.json]

Workloads (device-resident audio from ``device_synth``, every input larger than the 126 MB L2):
  c2        1024 stereo streams x 60 s at 48 kHz, one push per iteration (reset before each)
  c3_tiles  8192 stereo streams x 10 min at 48 kHz in 4 s time tiles with carried state (one 12.6 GB tile
            buffer pushed 150 times: the timing does not depend on the samples)
  c5_96k    64 streams x 8 channels x 30 s at 96 kHz, explicit weights, one push per iteration
Reported per workload: ms per push (CUDA events around the pushes after warm-up), stream-seconds per second,
the algorithmic bytes (4 B per input sample read, plus the series, peaks and state written) over the push time
as a share of the 7.7 TB/s HBM3e data-sheet peak, and the worst |GPU - float64 oracle| over 16 streams.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "audio-analyzer-omega_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

HBM_PEAK_BPS = 7.7e12
W_71 = [1.0, 1.0, 1.0, 0.0, 1.41, 1.41, 1.0, 1.0]


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def push_bytes(meter, n_rows, n):
    """Algorithmic bytes of one push: samples read + M/S series, peaks and carried state written."""
    steps = n // meter.sub + 1
    return 4 * n_rows * n + 2 * 4 * meter.n_streams * steps + 4 * n_rows + 8 * meter.n_streams * meter._h.state_doubles


def oracle_check(meter_series_m, meter_series_s, summary, x16, fs, weights):
    from oracle import bs1770_np as B
    ref = B.program_loudness(x16, fs, weights)
    worst = {}
    for key, got in (("momentary", meter_series_m), ("short_term", meter_series_s)):
        r = ref[key]
        assert np.array_equal(np.isnan(got), np.isnan(r)) and np.array_equal(np.isneginf(got), np.isneginf(r)), key
        sel = np.isfinite(r) & (r > -70.0)
        worst[key] = float(np.abs(got[sel] - r[sel]).max())
    for key in ("integrated", "lra"):
        g, r = summary[key][:16].astype(np.float64), ref[key]
        f = np.isfinite(r)
        assert np.array_equal(np.isfinite(g), f), key
        worst[key] = float(np.abs(g[f] - r[f]).max()) if f.any() else 0.0
    worst["pass_0.01_LU"] = bool(max(worst.values()) <= 0.01)
    return worst


def time_pushes(torch, fn, warmup, steps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_resident(torch, name, n_streams, n_ch, seconds, fs, weights, warmup, steps):
    from omega4_b200.batch.driver import device_synth
    from omega4_b200.loudness import LoudnessMeter
    n = int(seconds * fs)
    x = device_synth(n_streams, n_ch, n, fs)
    meter = LoudnessMeter(fs, weights, n_streams, max_seconds=seconds)

    def one():
        meter.reset()
        meter.push(x)

    ms = time_pushes(torch, one, warmup, steps)
    summ = meter.summary()
    m16 = meter.momentary[:16].cpu().numpy().astype(np.float64)
    s16 = meter.short_term[:16].cpu().numpy().astype(np.float64)
    x16 = x[:16 * n_ch].cpu().numpy().reshape(16, n_ch, n)
    from omega4_b200.tables import bs1770_channel_weights
    worst = oracle_check(m16, s16, summ, x16, fs, bs1770_channel_weights(weights, n_ch))
    b = push_bytes(meter, n_streams * n_ch, n)
    rec = {"workload": name, "streams": n_streams, "channels": n_ch, "seconds": seconds, "sample_rate": fs,
           "pushes_timed": steps, "ms_per_push": ms, "stream_seconds_per_s": n_streams * seconds / (ms / 1e3),
           "algorithmic_bytes": b, "achieved_GBps": b / (ms / 1e3) / 1e9,
           "hbm_share": b / (ms / 1e3) / HBM_PEAK_BPS, "oracle_worst_LU_16_streams": worst}
    del x
    torch.cuda.empty_cache()
    return rec, (m16, s16, summ)


def bench_tiles(torch, warmup, steps):
    """8192 stereo streams, 10 min in 4 s tiles with carried state; times the whole 150-tile pass."""
    from omega4_b200.batch.driver import device_synth
    from omega4_b200.loudness import LoudnessMeter
    fs, n_streams, tile_s, total_s = 48000, 8192, 4.0, 600.0
    n = int(tile_s * fs)
    x = device_synth(n_streams, 2, n, fs)
    meter = LoudnessMeter(fs, "stereo", n_streams, max_seconds=total_s)
    n_tiles = int(total_s / tile_s)

    def whole():
        meter.reset()
        for _ in range(n_tiles):
            meter.push(x)

    ms = time_pushes(torch, whole, max(1, warmup // 3), max(1, steps // 5))
    # the same tile pushed 150 times versus one push of the tile repeated: carried state across tiles
    summ = meter.summary()
    m16 = meter.momentary[:16].cpu().numpy().astype(np.float64)
    x16 = np.tile(x[:32].cpu().numpy().reshape(16, 2, n), (1, 1, 15))         # the first 60 s of the stream
    from oracle import bs1770_np as B
    ref = B.program_loudness(x16, fs, [1.0, 1.0])
    sel = np.isfinite(ref["momentary"]) & (ref["momentary"] > -70.0)
    worst_m = float(np.abs(m16[:, :600][sel] - ref["momentary"][sel]).max())
    b = push_bytes(meter, 2 * n_streams, n)
    per_push = ms / n_tiles
    rec = {"workload": "c3_tiles", "streams": n_streams, "channels": 2, "seconds": total_s, "tile_seconds": tile_s,
           "sample_rate": fs, "pushes_timed": n_tiles * max(1, steps // 5), "ms_per_push": per_push,
           "ms_per_10_min_pass": ms, "stream_seconds_per_s": n_streams * total_s / (ms / 1e3),
           "algorithmic_bytes": b, "achieved_GBps": b / (per_push / 1e3) / 1e9,
           "hbm_share": b / (per_push / 1e3) / HBM_PEAK_BPS,
           "oracle_worst_LU_16_streams": {"momentary_first_60_s": worst_m, "pass_0.01_LU": worst_m <= 0.01}}
    del x
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_loudness_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU fallback")
    res = {"card": card_info(), "torch_device": torch.cuda.get_device_name(0), "hbm_peak_Bps_datasheet": HBM_PEAK_BPS,
           "workloads": []}
    rec, _ = bench_resident(torch, "c2", 1024, 2, 60.0, 48000, "stereo", args.warmup, args.steps)
    res["workloads"].append(rec)
    res["workloads"].append(bench_tiles(torch, args.warmup, args.steps))
    rec, _ = bench_resident(torch, "c5_96k", 64, 8, 30.0, 96000, W_71, args.warmup, args.steps)
    res["workloads"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for w in res["workloads"]:
        print(f"{w['workload']:9s} {w['ms_per_push']:8.3f} ms/push  {w['stream_seconds_per_s'] / 1e6:8.3f} M stream-s/s  "
              f"{w['achieved_GBps']:7.0f} GB/s ({100 * w['hbm_share']:.1f} % of HBM peak)  oracle {w['oracle_worst_LU_16_streams']}")
    print("card:", res["card"])


if __name__ == "__main__":
    main()

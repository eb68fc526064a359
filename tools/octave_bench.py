"""Throughput of the one-third-octave band-level path (omega4_b200.octave) on one GPU, with an oracle check.

    python tools/octave_bench.py [--warmup 3] [--steps 10] [--out profiles/r04_octave_bench.json]

Workloads (device-resident audio from ``device_synth``, every input larger than the 126 MB L2):
  c2        1024 stereo streams (2048 rows) x 60 s at 48 kHz, one push per iteration (reset before each)
  c3_tiles  8192 stereo streams (16384 rows) at 48 kHz in 4 s tiles with carried state: warm-up and timed
            pushes continue one stream (the same 12.6 GB tile buffer each time: the timing does not depend on
            the samples)
  c5_96k    64 streams x 8 channels (512 rows) x 30 s at 96 kHz, one push per iteration
Reported per workload: ms per push (CUDA events around the timed pushes), stream-seconds per second; the float64
warp instructions per clock per SM, from the operation count of the kernel's inner loop (below) at the card's
maximum SM clock read in the same run, against the 1.79-1.84 warp-DFMA/clk/SM this card's pipes sustain
(profiles/r01_fp_pipes_microbench.txt); the algorithmic bytes over the push time as a share of the 7.7 TB/s
HBM3e data-sheet peak; and the worst |GPU - float64 oracle| over the first 16 rows.
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
PIPE_WARP_DFMA_PER_CLK_SM = (1.79, 1.84)
#: float64 warp instructions per row and sample in octave_kernel's inner loop: every lane runs three sections of
#: 1 DADD + 2 DFMA and one DFMA for the energy, so the warp issues 10 float64 instructions per sample of its row
FP64_WARP_INSTR_PER_SAMPLE = 10
ORACLE_ROWS = 16


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def max_sm_clock_hz(card: str):
    try:
        return float(card.split(",")[2].strip().split()[0]) * 1e6
    except (IndexError, ValueError):
        return None


def push_bytes(meter, n):
    """Algorithmic bytes of one push: samples read, block levels written, carried state read and written,
    Leq and Lmax written."""
    cols = meter.n_bands + 1
    steps = n // meter.sub + 1
    return meter.n_rows * (4 * n + 4 * steps * cols + 2 * 8 * meter._h.state_doubles + 2 * 4 * cols)


def oracle_worst(levels, leq, lmax, x, fs):
    """Worst |GPU - oracle| (dB) over block levels >= -150 dBFS, Leq and Lmax, with the -inf patterns checked."""
    from oracle import octave_np as O
    ref = O.band_levels(x, fs)
    worst = {}
    for key, got, floor in (("levels", levels, -150.0), ("leq", leq, -np.inf), ("max_level", lmax, -np.inf)):
        r = ref[key]
        assert np.array_equal(np.isneginf(got), np.isneginf(r)), key
        sel = np.isfinite(r) & (r >= floor)
        worst[key] = float(np.abs(got[sel].astype(np.float64) - r[sel]).max())
    worst["pass_1e-4_dB"] = bool(max(worst.values()) <= 1e-4)
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


def record(torch, name, meter, n_streams, n_ch, n, seconds_per_push, ms, clock_hz, worst, extra=None):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = n_streams * n_ch
    b = push_bytes(meter, n)
    rec = {"workload": name, "streams": n_streams, "channels": n_ch, "rows": rows, "bands": meter.n_bands,
           "sample_rate": meter.sample_rate, "seconds_per_push": seconds_per_push, "ms_per_push": ms,
           "stream_seconds_per_s": n_streams * seconds_per_push / (ms / 1e3),
           "warps_per_sm": rows / sms, "algorithmic_bytes": b, "achieved_GBps": b / (ms / 1e3) / 1e9,
           "hbm_share": b / (ms / 1e3) / HBM_PEAK_BPS, "oracle_rows": ORACLE_ROWS, "oracle_worst_dB": worst}
    fp64 = rows * n * FP64_WARP_INSTR_PER_SAMPLE
    rec["fp64_warp_instr"] = fp64
    if clock_hz:
        rec["fp64_warp_instr_per_clk_per_sm"] = fp64 / (ms / 1e3) / clock_hz / sms
        rec["share_of_pipe_rate"] = rec["fp64_warp_instr_per_clk_per_sm"] / PIPE_WARP_DFMA_PER_CLK_SM[1]
    rec.update(extra or {})
    return rec


def bench_resident(torch, name, n_streams, n_ch, seconds, fs, warmup, steps, clock_hz):
    from omega4_b200.batch.driver import device_synth
    from omega4_b200.octave import ThirdOctaveMeter
    n = int(seconds * fs)
    x = device_synth(n_streams, n_ch, n, fs)
    meter = ThirdOctaveMeter(fs, n_streams * n_ch, max_seconds=seconds)

    def one():
        meter.reset()
        meter.push(x)

    ms = time_pushes(torch, one, warmup, steps)
    worst = oracle_worst(meter.levels[:ORACLE_ROWS].cpu().numpy(), meter.leq[:ORACLE_ROWS].cpu().numpy(),
                         meter.max_level[:ORACLE_ROWS].cpu().numpy(), x[:ORACLE_ROWS].cpu().numpy(), fs)
    rec = record(torch, name, meter, n_streams, n_ch, n, seconds, ms, clock_hz, worst)
    meter.close()
    del x, meter
    torch.cuda.empty_cache()
    return rec


def bench_tiles(torch, warmup, steps, clock_hz):
    """8192 stereo streams in 4 s tiles; warm-up and timed pushes all continue the same streams."""
    from omega4_b200.batch.driver import device_synth
    from omega4_b200.octave import ThirdOctaveMeter
    fs, n_streams, tile_s = 48000, 8192, 4.0
    n = int(tile_s * fs)
    x = device_synth(n_streams, 2, n, fs)
    meter = ThirdOctaveMeter(fs, 2 * n_streams, max_seconds=tile_s * (warmup + steps))
    ms = time_pushes(torch, lambda: meter.push(x), warmup, steps)
    # carried state across tiles: the same tile pushed warmup + steps times against one oracle pass over them
    x16 = np.tile(x[:ORACLE_ROWS].cpu().numpy(), (1, warmup + steps))
    worst = oracle_worst(meter.levels[:ORACLE_ROWS].cpu().numpy(), meter.leq[:ORACLE_ROWS].cpu().numpy(),
                         meter.max_level[:ORACLE_ROWS].cpu().numpy(), x16, fs)
    rec = record(torch, "c3_tiles", meter, n_streams, 2, n, tile_s, ms, clock_hz, worst,
                 {"pushes_carried": warmup + steps, "stream_seconds_per_pass_of_10_min": 600.0,
                  "s_per_10_min_pass": ms / 1e3 * 600.0 / tile_s})
    meter.close()
    del x, meter
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_octave_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no CPU fallback")
    card = card_info()
    clock = max_sm_clock_hz(card)
    res = {"card": card, "torch_device": torch.cuda.get_device_name(0),
           "sm_count": torch.cuda.get_device_properties(0).multi_processor_count,
           "max_sm_clock_hz": clock, "hbm_peak_Bps_datasheet": HBM_PEAK_BPS,
           "pipe_warp_dfma_per_clk_sm_measured": PIPE_WARP_DFMA_PER_CLK_SM,
           "fp64_warp_instr_per_row_sample": FP64_WARP_INSTR_PER_SAMPLE, "warmup": args.warmup, "steps": args.steps,
           "workloads": []}
    res["workloads"].append(bench_resident(torch, "c2", 1024, 2, 60.0, 48000, args.warmup, args.steps, clock))
    res["workloads"].append(bench_tiles(torch, args.warmup, args.steps, clock))
    res["workloads"].append(bench_resident(torch, "c5_96k", 64, 8, 30.0, 96000, args.warmup, args.steps, clock))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for w in res["workloads"]:
        print(f"{w['workload']:9s} {w['ms_per_push']:8.2f} ms/push  {w['stream_seconds_per_s'] / 1e3:8.1f} k stream-s/s  "
              f"{w.get('fp64_warp_instr_per_clk_per_sm', float('nan')):.2f} fp64 warp-instr/clk/SM  "
              f"{100 * w['hbm_share']:.2f} % of HBM peak  oracle {w['oracle_worst_dB']}")
    print("card:", res["card"])


if __name__ == "__main__":
    main()

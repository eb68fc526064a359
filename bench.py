#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload config2|config3|config5]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): stream-seconds of 48 kHz stereo analysed per second through the full
multi-resolution FFT (8192/4096/2048/1024, hop 512) + combine + LUFS (M/S/I/LRA) + 4x true peak
pipeline.  Default workload = BASELINE config[2]: 1024 concurrent stereo streams x 60 s per GPU (weak
scaling: every rank analyses its own 1024 streams -- streams are independent, no data-path collective).
--workload config3 = BASELINE config[3] as written: 10-minute streams through StreamBatch time tiles with
carried state (weak: --streams per GPU; strong: --total-streams 8192 split over the ranks);
--workload config5 = BASELINE config[4]'s shape (96 kHz, 8 channels, six resolutions up to 32768).

One step = one pass of the whole path over that batch.  Printed JSON line (rank 0):
  value         device-resident throughput (inputs already in HBM), CUDA events, max over ranks
  e2e           same metric through the C ABI with HOST (pinned) buffers: H2D of every sample (the capture
                side's s16le wire format, omega4/audio/capture.py:571-574) and D2H of every result row
                (combined spectrum + meters) inside the timed region; e2e_variants: other result sets
  roofline      dominant kernel vs the measured HBM peak (this path is fp32-issue bound: see
                DESIGN.md section 5; roofline_fp32 gives the compute-side fractions)
  cpu_baseline  the reference's numpy/scipy CPU path (oracle PORT, oracle/ref_port.py) on this box's host cores
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True            # the benchmark leaves the tree as it found it (no __pycache__)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "audio-analyzer-omega_b200"))

METRIC = "stream-seconds of 48 kHz stereo analysed/sec (multi-res FFT+LUFS+TP)"
UNIT = "stream-s/s"
SR, HOP, T_BINS, CHANNELS = 48000, 512, 512, 2
B_ALG_PER_HOP = 2048 + 2048 + 20          # SURVEY.md section 8d, fused-output mode: 512 f32 in, 512 f32 + 5 f32 out
FLOP_PER_HOP = 0.9e6                      # SURVEY.md section 8d nominal estimate (all four FFTs + meters on CUDA cores)
FLOP_TENSOR_FFT = 266240 + 122880         # the 8192 + 4096 FFTs of that estimate: now a tensor-core GEMM instead
TENSOR_FLOP_PER_HOP = 3 * 2 * 960 * 512   # split-precision hop-block GEMM (three products): 960 columns x 512 samples per hop block
FP32_PEAK_TFLOPS = 70.8                   # measured FFMA peak on this pool's B200 (profiles/r01_fp_pipes_microbench.txt:
                                          # 121.7 lanes/clk/SM x 148 SMs x 1.965 GHz x 2); nominal 75
DUMP_ROWS = 16384                         # --dump-outputs: 16384 x (512 + 5) float32 = 34 MB at most


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# host placement: pin the rank (and the pages it is about to pin) to the GPU's NUMA node
# ---------------------------------------------------------------------------------------------------------
def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(local_rank, local_world):
    """Bind this process and its future page allocations to the NUMA node of GPU `local_rank` BEFORE any pinned
    buffer is allocated (cudaHostAlloc pins the pages where they are first touched).  Returns what was done; on a
    VM that exposes no topology (numa_node = -1, one node) there is nothing to bind to and the CPUs are only
    partitioned between the ranks so that their copy threads do not share cores."""
    info = {"node": None, "cpus": None, "mempolicy": None, "how": None}
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{getattr(p, 'pci_domain_id', 0):04x}:{p.pci_bus_id:02x}:{getattr(p, 'pci_device_id', 0):02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        info["pci"] = bus
    except Exception as e:
        info["how"] = f"GPU PCI address / numa_node not readable ({type(e).__name__})"
        node = -1
    all_cpus = sorted(os.sched_getaffinity(0))
    if node >= 0 and os.path.isdir(f"/sys/devices/system/node/node{node}"):
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = sorted(_parse_cpulist(f.read()) & set(all_cpus))
        # ranks that share a node split its CPUs
        if cpus:
            os.sched_setaffinity(0, cpus)
        info.update(node=node, cpus=len(cpus), how="sched_setaffinity to the GPU's node")
        try:                                                  # set_mempolicy(MPOL_PREFERRED, node): x86_64 syscall 238
            libc = ctypes.CDLL(None, use_errno=True)
            mask = ctypes.c_ulong(1 << node)
            rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(64))
            info["mempolicy"] = "preferred" if rc == 0 else f"set_mempolicy failed (errno {ctypes.get_errno()})"
        except Exception as e:
            info["mempolicy"] = f"unavailable ({type(e).__name__})"
    else:
        per = max(1, len(all_cpus) // max(1, local_world))
        mine = all_cpus[local_rank * per:(local_rank + 1) * per] or all_cpus
        if local_world > 1:
            os.sched_setaffinity(0, mine)
        info.update(node=node, cpus=len(mine), how=info["how"] or "no NUMA topology exposed (numa_node = -1): CPUs partitioned between the ranks only")
    return info


def dump_outputs(out_dir, comb, met):
    """Write the same seeded sample of rows (row = channel * n_hops + hop) of the step's outputs ``comb``
    [n_ch, n_hops, T] and ``met`` [n_ch, n_hops, 5] to out_dir/combined.npy and out_dir/meters.npy."""
    import numpy as np
    import torch
    n_rows = comb.shape[0] * comb.shape[1]
    rows = np.sort(np.random.default_rng(0).choice(n_rows, min(DUMP_ROWS, n_rows), replace=False))
    idx = torch.from_numpy(rows).to(comb.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "combined.npy"), comb.reshape(n_rows, -1)[idx].cpu().numpy())
    np.save(os.path.join(out_dir, "meters.npy"), met.reshape(n_rows, -1)[idx].cpu().numpy())


def cpu_baseline(sample_seconds, streams=None, repeat=1):
    """Times oracle/ref_port.py (the reference's per-hop numpy/scipy path, a PORT pinned to the oracle) in a fresh
    interpreter on all host cores; returns (list of results, cores, streams)."""
    cores = os.cpu_count() or 1
    n = streams or cores
    cmd = [sys.executable, "-m", "oracle.ref_port", "--streams", str(n), "--seconds", str(sample_seconds),
           "--processes", str(cores), "--repeat", str(repeat)]
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1", PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    if out.returncode != 0:
        raise RuntimeError("cpu baseline failed: " + out.stderr[-2000:])
    return json.loads(out.stdout.strip().splitlines()[-1]), cores, n


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle PORT: the reference is
    Python and is not on the GPU box) on the host cores, same metric and config."""
    if rank != 0:
        return
    secs = args.cpu_seconds
    res, cores, n = cpu_baseline(secs, repeat=args.warmup + args.steps)
    timed = res[args.warmup:]
    wall = sum(r["wall_s"] for r in timed)
    value = sum(r["stream_seconds"] for r in timed) / wall
    sample = f"{n} stereo streams x {secs:g} s per step, {cores} processes (OMP_NUM_THREADS=1), {cpu_model()}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, len(timed)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 FFT / f64 meters (numpy, scipy)", "data": "synthetic",
        "config": {"workload": "BASELINE config[2] shape: stereo 48 kHz streams, 4 resolutions 8192/4096/2048/1024, hop 512, "
                               "512 target bins, LUFS M/S/I/LRA + 4x true peak; bounded sample per step", "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "cpu": cpu_model()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=1024, help="streams per GPU (config[2]: 1024)")
    ap.add_argument("--total-streams", type=int, default=0,
                    help="strong scaling: this many streams in total, split evenly over the ranks (overrides --streams)")
    ap.add_argument("--seconds", type=int, default=0, help="seconds per stream (default: 60; config3: 600)")
    ap.add_argument("--e2e-streams", type=int, default=1024,
                    help="streams per host-buffer call of the e2e leg (halved until the pinned buffers can be allocated)")
    ap.add_argument("--e2e-variants", default="bars,meters",
                    help="other result sets timed after the headline e2e (comma list of bars, meters, f32; empty = none)")
    ap.add_argument("--cpu-seconds", type=float, default=60.0,
                    help="seconds per stream of the CPU baseline sample (one stream per host core; 60 s = the workload's stream length)")
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config5"],
                    help="config2 (default, the metric's configuration): 48 kHz stereo x 60 s, 8192/4096/2048/1024; "
                         "config3: the same streams x 10 min through StreamBatch time tiles with carried state (BASELINE configs[3]); "
                         "config5: 96 kHz 8-channel (7.1) streams, six resolutions 32768 .. 1024 (BASELINE configs[4] shape)")
    ap.add_argument("--flags", type=int, default=0, help="extra omega4_analyze flags (developer A/B runs, e.g. 64 = OMEGA4_FLAG_SERIAL_STATS)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0; config3: its last time "
                         "tile) as DIR/combined.npy float32 [R, 512] and DIR/meters.npy float32 [R, 5]: the same "
                         f"R <= {DUMP_ROWS} (channel, hop) rows of both, drawn with a fixed seed.  The input signal is "
                         "seeded as well, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if args.impl == "reference":
        return run_reference(args, rank)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    import torch.distributed as dist
    from omega4_b200 import _native as N
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS, CONFIG5_96K
    from omega4_b200.batch.driver import device_synth, StreamBatch
    from omega4_b200.batch.partition import gather_rows, final_rows

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU arm)")
    numa = {"how": "disabled (--no-numa)"} if args.no_numa else bind_to_gpu_numa_node(local, local_world)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    global SR, CHANNELS
    configs, wl_name = BASELINE_CONFIGS, "BASELINE config[2]"
    seconds = args.seconds or 60
    if args.workload == "config5":
        SR, CHANNELS, configs, wl_name = 96000, 8, CONFIG5_96K, "BASELINE configs[4] shape (96 kHz, 8 channels, 6 resolutions)"
        args.no_cpu = True                       # the CPU leg times the metric's configuration only
    if args.workload == "config3":
        wl_name, seconds = "BASELINE configs[3]", args.seconds or 600
    scaling = "weak"
    if args.total_streams:
        if args.total_streams % world:
            raise SystemExit("--total-streams must be a multiple of the number of ranks")
        args.streams, scaling = args.total_streams // world, "strong"
    n_streams, n_ch = args.streams, args.streams * CHANNELS
    total_hops = seconds * SR // HOP
    plan = AnalysisPlan(SR, configs, T_BINS, device=local)
    first_stream = rank * n_streams

    # time tiling: config2 / config5 keep the whole clip resident (one tile); config3 walks 10 minutes in tiles of
    # at most 60 s sized so that one tile's input + outputs stay below ~60 GB of the 180 GB
    tiled = args.workload == "config3"
    tile_hops = total_hops
    if tiled:
        per_ch_hop = HOP * 4 + T_BINS * 4 + 20 + 50 * 8 + 16
        tile_hops = int(min(60 * SR // HOP, max(64, 60e9 // (n_ch * per_ch_hop))))
    n_tiles = (total_hops + tile_hops - 1) // tile_hops
    tile_sizes = [min(tile_hops, total_hops - i * tile_hops) for i in range(n_tiles)]
    n_samples = tile_hops * HOP
    sb = None
    if tiled:
        # the stream is the tile's 60 s (or shorter) clip repeated: generated once into the tile view, where it stays
        sb = StreamBatch(plan, n_ch, tile_hops)
        x = sb.tile_view(tile_hops)
        device_synth(n_streams, CHANNELS, n_samples, SR, first_stream=first_stream, device=local, out=x)
    else:
        x = device_synth(n_streams, CHANNELS, n_samples, SR, first_stream=first_stream, device=local)
    comb = torch.empty((n_ch, tile_hops, T_BINS), dtype=torch.float32, device=dev)
    met = torch.empty((n_ch, tile_hops, N.N_METERS), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(flags=0):
        if not tiled:
            plan.analyze_device(x, total_hops, 0, combined=comb, meters=met, flags=flags | args.flags | N.FLAG_FRESH_METERS)
            return
        sb.hist, sb.hops_done = 0, 0
        for i, n in enumerate(tile_sizes):
            last = i == n_tiles - 1
            sb.push(n, combined=comb[:, :n] if n == tile_hops else comb.view(-1)[:n_ch * n * T_BINS].view(n_ch, n, T_BINS),
                    meters=met[:, :n] if n == tile_hops else met.view(-1)[:n_ch * n * N.N_METERS].view(n_ch, n, N.N_METERS),
                    flags=args.flags | (flags if last else 0))

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    try:
        launches0 = plan.launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ktimes = {}
        ev0.record()
        for _ in range(args.steps):
            step(N.FLAG_TIME_KERNELS)            # the library brackets each kernel with events on this stream
        ev1.record()
        barrier()
        # kernel times of the last timed step's (last tile's) call (events of earlier calls are overwritten; same launches)
        for name, ms in plan.kernel_times():
            ktimes[name] = ms
        launches = plan.launches - launches0

        t_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    finally:                                     # a failed step must not leave nvidia-smi running
        clocks = sampler.stop() if rank == 0 else None
    total_ms = float(t_ms[0])
    ms_per_step = total_ms / args.steps
    stream_seconds_per_step = n_streams * seconds * world
    value = stream_seconds_per_step / (ms_per_step / 1e3)

    # what the last timed step computed: the last tile's rows (config3's last tile may be shorter than the buffers)
    last_n = tile_sizes[-1]
    comb_out = comb if last_n == tile_hops else comb.view(-1)[:n_ch * last_n * T_BINS].view(n_ch, last_n, T_BINS)
    met_out = met if last_n == tile_hops else met.view(-1)[:n_ch * last_n * N.N_METERS].view(n_ch, last_n, N.N_METERS)
    if args.dump_outputs and rank == 0:          # before the e2e leg below reuses comb / met
        dump_outputs(args.dump_outputs, comb_out, met_out)

    # the only collective of the whole path: gather the final per-stream rows (after the timed region):
    # the meters of the last hop + the last combined spectrum of every channel
    met_last = met_out[:, -1, :]
    comb_last = comb_out[:, -1, :]
    rows = torch.cat([met_last, comb_last], dim=1).reshape(n_streams, CHANNELS, N.N_METERS + T_BINS).contiguous()
    allrows = gather_rows(rows, n_streams * world) if world > 1 else rows
    checksum = float(allrows[..., :N.N_METERS].double().sum())

    # multi-GPU result parity: rank 0 re-analyses streams another rank owns and compares the gathered rows bit for bit
    mgpu = None
    if world > 1 and rank == 0:
        k = min(2, n_streams)
        owner = world - 1
        fs = owner * n_streams
        if tiled:
            sb2 = StreamBatch(plan, k * CHANNELS, tile_hops)
            device_synth(k, CHANNELS, n_samples, SR, first_stream=fs, device=local, out=sb2.tile_view(tile_hops))
            c2 = torch.empty((k * CHANNELS, tile_hops, T_BINS), device=dev)
            m2 = torch.empty((k * CHANNELS, tile_hops, N.N_METERS), device=dev)
            for n in tile_sizes:
                sb2.push(n, combined=c2.view(-1)[:k * CHANNELS * n * T_BINS].view(k * CHANNELS, n, T_BINS),
                         meters=m2.view(-1)[:k * CHANNELS * n * N.N_METERS].view(k * CHANNELS, n, N.N_METERS), flags=args.flags)
            c2 = c2.view(-1)[:k * CHANNELS * last_n * T_BINS].view(k * CHANNELS, last_n, T_BINS)
            m2 = m2.view(-1)[:k * CHANNELS * last_n * N.N_METERS].view(k * CHANNELS, last_n, N.N_METERS)
            del sb2
        else:
            x2 = device_synth(k, CHANNELS, n_samples, SR, first_stream=fs, device=local)
            c2 = torch.empty((k * CHANNELS, total_hops, T_BINS), device=dev)
            m2 = torch.empty((k * CHANNELS, total_hops, N.N_METERS), device=dev)
            plan.analyze_device(x2, total_hops, 0, combined=c2, meters=m2, flags=args.flags | N.FLAG_FRESH_METERS)
        torch.cuda.synchronize()
        mine = torch.cat([m2[:, -1, :], c2[:, -1, :]], dim=1).reshape(k, CHANNELS, -1)
        theirs = allrows[fs:fs + k]
        mgpu = {"streams": [fs, fs + k - 1], "owner_rank": owner, "recomputed_on_rank": 0,
                "meters_bit_identical": bool(torch.equal(mine[..., :N.N_METERS], theirs[..., :N.N_METERS])),
                "combined_bit_identical": bool(torch.equal(mine[..., N.N_METERS:], theirs[..., N.N_METERS:]))}
        del c2, m2

    # ---------------- end-of-stream rows of one channel against the oracle (config3: the 10-minute tiled stream)
    oracle_check = None
    if tiled and rank == 0:
        from oracle import oracle_np as O
        tail_hops = 3600 + 64
        P = n_samples                                               # the stream is periodic with the tile's clip
        end = total_hops * HOP
        beg = end - tail_hops * HOP - max(c[1] for c in configs)
        clip = x[0].cpu().numpy()
        idx = (np.arange(beg, end) % P)
        ref = O.analyze_channel(clip[idx], SR, O.BASELINE_CONFIGS)
        got_m = met_last[0].cpu().numpy().astype(np.float64)
        got_c = comb_last[0].cpu().numpy().astype(np.float64)
        rc_ = ref["combined"][-1].astype(np.float64)
        sig = rc_ >= rc_.max() * 1e-4
        oracle_check = {"channel": 0, "hops_replayed_by_the_oracle": tail_hops,
                        "meters_abs_err": [float(v) for v in np.abs(got_m - ref["meters"][-1])],
                        "combined_max_db_err_within_80dB": float(np.abs(20 * np.log10(np.maximum(got_c[sig], 1e-30)) - 20 * np.log10(rc_[sig])).max()),
                        "pass": bool(np.abs(got_m - ref["meters"][-1])[:4].max() <= 0.01 and abs(got_m[4] - ref["meters"][-1][4]) <= 0.05)}

    # ---------------- SURVEY section 8f rows, timed separately (not part of the headline metric)
    next_rows = {}
    post = None
    try:
        from omega4_b200.app.spectrum_post import SpectrumPostProcessor
        if args.workload == "config5":
            raise RuntimeError("timed for 48 kHz workloads only")
        post = SpectrumPostProcessor(T_BINS, SR, 2048, device=local)
        post._ensure()
        bars = torch.empty((n_ch, tile_hops, post.n_valid), dtype=torch.float32, device=dev)
        post.process_device(comb, bars)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        post.process_device(comb, bars)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        next_rows["app_post_processing"] = {"ms": ms, "bars_per_frame": post.n_valid,
                                            "gbs": (comb.numel() + bars.numel()) * 4 / (ms / 1e3) / 1e9,
                                            "frac_hbm": (comb.numel() + bars.numel()) * 4 / (ms / 1e3) / 1e9 / float(measured_peaks()[0].get("hbm_gbs", 6650.0))}
        del bars
    except Exception as e:                       # never let an auxiliary row break the headline line
        next_rows["app_post_processing"] = {"error": str(e)}

    # ---------------- e2e: host (pinned) buffers through the C ABI, int16 wire format in, result rows out
    e2e, e2e_variants = None, {}
    if not args.no_e2e:
        es = min(args.e2e_streams, n_streams)
        per_stream = CHANNELS * (n_samples * 2 + tile_hops * (T_BINS + N.N_METERS) * 4)
        try:                                          # never pin more than ~35 % of the free host memory per node
            import psutil
            avail = psutil.virtual_memory().available
            while es > 16 and es * per_stream * local_world > 0.35 * avail:
                es //= 2
        except Exception:
            pass
        hist_cap = sb.hist_cap if tiled else 0
        hx = hcomb = hmet = None
        while True:                                   # biggest pinned host batch this box can give us
            ech = es * CHANNELS
            try:
                hx = torch.empty((es, hist_cap + n_samples, CHANNELS), dtype=torch.int16, pin_memory=True)
                hcomb = torch.empty((ech, tile_hops, T_BINS), dtype=torch.float32, pin_memory=True)
                hmet = torch.empty((ech, tile_hops, N.N_METERS), dtype=torch.float32, pin_memory=True)
                break
            except RuntimeError:
                hx = hcomb = hmet = None
                if es <= 16:
                    raise
                es //= 2
        calls = (n_streams + es - 1) // es
        # quantise the resident clip to the wire format, stream by stream (x = int16 / 32768 on the way back in)
        for s0 in range(0, es, 64):
            s1 = min(es, s0 + 64)
            blk = x[s0 * CHANNELS:s1 * CHANNELS].reshape(s1 - s0, CHANNELS, n_samples)
            q = (blk.clamp(-1.0, 1.0) * 32767.0).round().to(torch.int16).permute(0, 2, 1).contiguous()
            hx[s0:s1, hist_cap:].copy_(q)
            if hist_cap:                              # periodic stream: the history of a tile is the clip's own tail
                hx[s0:s1, :hist_cap].copy_(q[:, n_samples - hist_cap:])
            del q, blk
        torch.cuda.synchronize()
        hstate = torch.zeros((ech, N.METER_STATE_DOUBLES), dtype=torch.float64, pin_memory=True) if tiled else None
        stride16 = hx.stride(0)
        base16 = hx.data_ptr() + hist_cap * CHANNELS * 2
        lib = N.lib()

        def run_e2e(kind):
            """One step through the C ABI with host buffers.  kind: full (combined + meters), bars (band_values +
            meters), meters (meters only); config3 walks the tiles with the meter state carried on the host."""
            for _ in range(calls):
                done = 0
                for i, n in enumerate(tile_sizes):
                    hist = min(hist_cap, done * HOP)
                    fl = N.FLAG_FRESH_METERS if i == 0 else 0
                    if kind == "bars":
                        plan.analyze_io(N.MEM_HOST, ech, n, stride16, frames_s16=base16, n_interleaved=CHANNELS, hist=hist,
                                        meters=hmet, meter_state=hstate, bars=post, band_values=hbars,
                                        bars_state=hbstate if tiled else None, flags=fl | (N.FLAG_FRESH_BARS if i == 0 else 0))
                    else:
                        rc = lib.omega4_analyze_s16(plan.handle, None, N.MEM_HOST, base16, stride16, es, CHANNELS, n, hist,
                                                    hcomb.data_ptr() if kind == "full" else None, None, hmet.data_ptr(), None, None,
                                                    hstate.data_ptr() if tiled else None, fl)
                        N.check(rc, "omega4_analyze_s16(host)")
                    done += n

        def time_e2e(kind, steps):
            run_e2e(kind)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                run_e2e(kind)
            barrier()
            et = torch.tensor([(time.perf_counter() - t0) / steps], device=dev)
            if world > 1:
                dist.all_reduce(et, op=dist.ReduceOp.MAX)
            return float(et[0])

        sum_hops = sum(tile_sizes)
        h2d = calls * es * CHANNELS * (sum_hops * HOP + (n_tiles - 1) * hist_cap) * 2 + \
            (calls * (n_tiles - 1) * ech * N.METER_STATE_DOUBLES * 8 if tiled else 0)
        d2h_meters = calls * ech * sum_hops * N.N_METERS * 4 + (calls * n_tiles * ech * N.METER_STATE_DOUBLES * 8 if tiled else 0)
        d2h_full = d2h_meters + calls * ech * sum_hops * T_BINS * 4
        t_full = time_e2e("full", args.steps)
        per_step_ss = calls * es * seconds * world
        e2e = {"value": per_step_ss / t_full, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full,
               "ms_per_step": 1e3 * t_full, "steps_timed": args.steps,
               "input": "interleaved int16 (s16le, the capture side's wire format; omega4_analyze_s16)",
               "results": "combined spectrum float32[512] + meters float32[5] per channel-hop",
               "bus_gbs_per_gpu": (h2d + d2h_full) / t_full / 1e9, "bus_gbs_all_gpus": (h2d + d2h_full) * world / t_full / 1e9,
               "host_buffers": f"{calls} calls x {es} streams x {seconds} s per step from the same pinned buffers"
                               + (f", {n_tiles} time tiles per call with the meter state carried on the host" if tiled else ""),
               "numa": numa}
        # parity of the host-buffer leg against a device-resident run of the same int16 frames: meters AND combined
        d16 = hx[:, hist_cap:].to(dev, non_blocking=True) if not tiled else None
        if d16 is not None:
            plan.analyze_s16_device(d16.view(es, -1), total_hops, CHANNELS, combined=comb[:ech], meters=met[:ech], flags=N.FLAG_FRESH_METERS)
            torch.cuda.synchronize()
            same_c, worst = True, 0.0
            for c0 in range(0, ech, 128):             # compare on the device, 128 channels at a time
                a_, b_ = hcomb[c0:c0 + 128].to(dev), comb[c0:c0 + 128]
                if not torch.equal(a_, b_):
                    same_c = False
                    worst = max(worst, float(((a_ - b_).abs() / (b_.amax(dim=2, keepdim=True) + 1e-30)).max()))
            # (transforms of more than 16 hop blocks -- config5's 32768 / 16384 -- complete their frames with several
            # float atomics per value: the summation order, hence the last bit, varies from run to run)
            e2e["parity_vs_resident"] = {"meters": bool(torch.equal(hmet.to(dev), met[:ech])), "combined": same_c,
                                         "combined_max_abs_diff_over_row_max": worst}
            del d16
        # other result sets / inputs, a few steps each
        for kind in [k for k in args.e2e_variants.split(",") if k]:
            vs = max(1, min(args.steps, 3))
            try:
                if kind == "bars":
                    if post is None:
                        raise RuntimeError("no bars object for this workload")
                    hbars = torch.empty((ech, tile_hops, post.n_valid), dtype=torch.float32, pin_memory=True)
                    hbstate = torch.zeros((ech, 1 + post.n_valid), dtype=torch.float32, pin_memory=True)
                    t = time_e2e("bars", vs)
                    d2h = d2h_meters + calls * ech * sum_hops * post.n_valid * 4
                    e2e_variants["bars"] = {"value": per_step_ss / t, "ms_per_step": 1e3 * t, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                            "results": f"band_values float32[{post.n_valid}] (omega4_main.py:1011-1056, fused behind the combine) + meters",
                                            "steps_timed": vs}
                    del hbars, hbstate
                elif kind == "meters":
                    t = time_e2e("meters", vs)
                    e2e_variants["meters"] = {"value": per_step_ss / t, "ms_per_step": 1e3 * t, "h2d_bytes_per_step": h2d,
                                              "d2h_bytes_per_step": d2h_meters, "results": "meters float32[5] only", "steps_timed": vs}
                elif kind == "f32" and not tiled:
                    hxf = torch.empty((ech, n_samples), dtype=torch.float32, pin_memory=True)
                    hxf.copy_(x[:ech])

                    def f32_step():
                        for _ in range(calls):
                            rc = lib.omega4_analyze(plan.handle, None, N.MEM_HOST, hxf.data_ptr(), n_samples, ech, total_hops, 0,
                                                    hcomb.data_ptr(), None, hmet.data_ptr(), None, None, None, 0)
                            N.check(rc, "omega4_analyze(host)")
                    f32_step()
                    barrier()
                    t0 = time.perf_counter()
                    for _ in range(vs):
                        f32_step()
                    barrier()
                    et = torch.tensor([(time.perf_counter() - t0) / vs], device=dev)
                    if world > 1:
                        dist.all_reduce(et, op=dist.ReduceOp.MAX)
                    t = float(et[0])
                    e2e_variants["f32"] = {"value": per_step_ss / t, "ms_per_step": 1e3 * t, "h2d_bytes_per_step": calls * hxf.numel() * 4,
                                           "d2h_bytes_per_step": d2h_full, "results": "float32 input rows (round 1's e2e leg)", "steps_timed": vs}
                    del hxf
            except Exception as e:
                e2e_variants[kind] = {"error": str(e)}
        del hx, hcomb, hmet
    if post is not None:
        post.close()

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        is48_wl = args.workload != "config5"
        ch_hops = n_ch * total_hops
        k_hops = n_ch * last_n                                        # channel-hops of the call the kernel times belong to
        # the statistics kernel runs on a side stream underneath the FFT kernels: its CUDA-event span is mostly waiting
        # for SM slots, so it only counts as the dominant kernel when it runs in line (OMEGA4_FLAG_SERIAL_STATS)
        cand = {k: v for k, v in ktimes.items() if k != "meter_stats" or (args.flags & N.FLAG_SERIAL_STATS)}
        dom = max(cand, key=cand.get) if cand else None
        roof = None
        if dom:
            # algorithmic bytes of the dominant kernel per launch: every input sample once + what it writes
            out_bytes = {"multires_fft_8192": 6 * 4, "multires_fft_4096": 20 * 4, "multires_fft_2048": 102 * 4,
                         "multires_fft_1024": 384 * 4, "true_peak": 8, "kweight_lufs": 8, "meter_stats": 20,
                         "blockdft_gemm": 128 * 4, "blockdft_tc_gemm": 50 * 8, "blockdft_asm_8192": 6 * 4,
                         "blockdft_asm_4096": 20 * 4, "blockdft_row_scale": 4}.get(dom, 0)
            if dom.startswith("multires_fft_") and not is48_wl:      # config5: target bins per resolution differ
                out_bytes = {"multires_fft_4096": 102 * 4, "multires_fft_2048": 179 * 4, "multires_fft_1024": 205 * 4}.get(dom, out_bytes)
            in_bytes = {"meter_stats": 16, "blockdft_asm_8192": 100 * 4, "blockdft_asm_4096": 400 * 4}.get(dom, HOP * 4)
            alg = k_hops * (in_bytes + out_bytes)
            ach = alg / (ktimes[dom] / 1e3) / 1e9
            traffic = None
            try:
                with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                    tj = json.load(f)
                if tj.get("kernel") == dom and tj.get("channel_hops") == k_hops:
                    traffic = tj.get("dram_bytes_per_launch")
            except Exception:
                pass
            # nominal arithmetic of the kernel per channel-hop (5 N log2 N per complex FFT, FMA = 2): the compute-side
            # view of the same kernel, next to the HBM view the contract asks for
            kflop = {"true_peak": 2 * 5 * 2048 * 11 + 3 * 2048 * 6, "kweight_lufs": 4 * 2080 * 14,
                     "multires_fft_2048": 5 * 1024 * 10 + 1024 * 12 + 2048, "multires_fft_1024": 5 * 512 * 9 + 512 * 12 + 1024,
                     "multires_fft_4096": 5 * 2048 * 11 + 2048 * 12 + 4096, "multires_fft_8192": 5 * 4096 * 12 + 4096 * 12 + 8192}.get(dom)
            fp32 = None
            if kflop:
                tf = k_hops * kflop / (ktimes[dom] / 1e3) / 1e12
                note = "FFT butterflies are additions, not FMAs: at 100 % issue this instruction mix reaches about half the FMA peak"
                if dom == "true_peak" and not (args.flags & N.FLAG_EXACT_TRUE_PEAK):
                    note += ("; the kernel's transforms run as half2 instructions, which occupy the FMA pipe at the float32 rate "
                             "per scalar operation (HFMA2 1.9 against FFMA 3.7 warp instructions per clock and SM, "
                             "profiles/r02l_f32x2_pipes.txt), so the nominal float32 count still measures the pipe")
                fp32 = {"flop_per_channel_hop": kflop, "achieved_tflops": tf, "peak_tflops_measured": FP32_PEAK_TFLOPS,
                        "frac": tf / FP32_PEAK_TFLOPS, "note": note}
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": traffic, "peak_source": peak_kind, "kernel_ms": ktimes[dom], "fp32": fp32,
                    "kernel_share_of_step": ktimes[dom] / sum(ktimes.values()),
                    "note": "fp32-issue bound by arithmetic (about 220 FLOP per compulsory byte): low HBM fraction is expected; "
                            "kernel_share_of_step is of the summed kernel times (the statistics kernel overlaps the FFT kernels)"}
        pipe_gbs = ch_hops * B_ALG_PER_HOP / (ms_per_step / 1e3) / 1e9
        step_s = ms_per_step / 1e3
        is48 = args.workload != "config5"
        line = {
            "metric": METRIC if is48 else METRIC.replace("48 kHz stereo", "96 kHz 8-channel"),
            "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f32 (FFT, combine, K-weighting in a float32 delta-form state, sample peaks of the true-peak meter; its four transforms per frame pair in f16x2; tensor-core GEMM on (hi, lo) half operands with fp32 accumulators for the few-bin resolutions) + f64 (meter statistics)",
            "data": "synthetic",
            "config": {"workload": f"{wl_name}: {n_streams} streams x {CHANNELS} ch x {seconds} s @{SR // 1000} kHz per GPU"
                                   + (f" ({n_streams * world} streams in total, strong scaling)" if scaling == "strong" else "")
                                   + f", resolutions {'/'.join(str(c[1]) for c in configs)}, hop 512, 512 target bins (fused output mode B), "
                                   "LUFS M/S/I/LRA + 4x true peak per hop"
                                   + (f"; {n_tiles} time tiles of <= {tile_hops} hops per step through StreamBatch, window history and "
                                      "meter deques carried between tiles, the tile's clip repeated (periodic stream, resident in HBM)" if tiled else ""),
                       "streams_per_gpu": n_streams, "seconds": seconds, "channels": CHANNELS, "time_tiles_per_step": n_tiles,
                       "channel_hops_per_step_per_gpu": ch_hops, "parallelism": f"streams sharded x{world}, no data-path collective",
                       "l2": f"inputs {x.numel()*4/1e9:.1f} GB + outputs {comb.numel()*4/1e9:.1f} GB per tile >> 126 MB L2 (no flush needed)"},
            "roofline": roof,
            "pipeline_hbm": {"algorithmic_bytes_per_channel_hop": B_ALG_PER_HOP, "achieved_gbs": pipe_gbs, "frac": pipe_gbs / hbm_peak},
            "kernel_ms": ktimes, "gpu_launches": launches, "clocks": clocks, "e2e": e2e, "e2e_variants": e2e_variants,
            "next_rows": next_rows, "final_rows_checksum": checksum, "multi_gpu_parity": mgpu, "oracle_check": oracle_check,
        }
        if is48:
            nominal = ch_hops * FLOP_PER_HOP / step_s / 1e12
            executed = ch_hops * (FLOP_PER_HOP - FLOP_TENSOR_FFT) / step_s / 1e12
            line["roofline_fp32"] = {
                "nominal": {"flop_per_channel_hop": FLOP_PER_HOP, "achieved_tflops": nominal, "frac": nominal / FP32_PEAK_TFLOPS,
                            "note": "SURVEY 8d's count, as if all four FFTs ran on the CUDA cores"},
                "executed_cuda_cores": {"flop_per_channel_hop": FLOP_PER_HOP - FLOP_TENSOR_FFT, "achieved_tflops": executed,
                                        "frac": executed / FP32_PEAK_TFLOPS,
                                        "note": "without the 8192 + 4096 FFTs, whose bins come from the tensor-core GEMM"},
                "tensor_cores": {"flop_per_channel_hop": TENSOR_FLOP_PER_HOP, "kind": "f16 (hi + lo / 2^11 split of row-scaled operands, three products, fp32 accumulators)",
                                 "achieved_tflops_in_kernel": (k_hops * TENSOR_FLOP_PER_HOP / (ktimes["blockdft_tc_gemm"] / 1e3) / 1e12)
                                 if ktimes.get("blockdft_tc_gemm") else None},
                "peak_tflops_measured": FP32_PEAK_TFLOPS,
                "frac": nominal / FP32_PEAK_TFLOPS}
        if world == 1 and not args.no_cpu:
            try:
                res, cores, n = cpu_baseline(args.cpu_seconds)
                line["cpu_baseline"] = {"value": res[0]["value"], "unit": UNIT, "cores": cores, "kind": "port", "cpu": cpu_model(),
                                        "sample": f"{n} stereo streams x {args.cpu_seconds:g} s, {cores} processes, OMP_NUM_THREADS=1, "
                                                  f"{res[0]['wall_s']:.1f} s wall (oracle/ref_port.py: a port of the reference's call structure, "
                                                  "pinned to the oracle; the reference itself is Python and does not travel to the GPU box)",
                                        "cpu_s_per_stream_second_per_core": res[0]["cpu_s_per_stream_second"]}
            except Exception as e:       # the GPU numbers stand on their own
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
        if mgpu and not (mgpu["meters_bit_identical"] and mgpu["combined_bit_identical"]):
            raise SystemExit("multi-GPU parity FAILED: gathered rows differ from the rows recomputed on rank 0")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

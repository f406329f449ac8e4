#!/usr/bin/env python3
"""bench.py -- channel-samples/s of the 4-slot EAX reverb chain (BASELINE.json metric).

One "step" = one 1024-frame block of the hot path (oalsfx_engine_mix: source encode + dry mix +
equalizer + chorus + echo + EAX reverb + output interleave, fused) over ALL streams of the rank.

Workload at N=1 = BASELINE.json configs[4] on one GPU ("cfg4": 65 536 independent stereo 48 kHz
streams, static default parameters) -- the configuration the metric and the north_star target are
quoted on.  With N>1 every rank runs the same 65 536 streams on its own GPU (streams shard with no
data-path collective: "weak" scaling); `value` is the whole-job aggregate.  The same line also carries
  configs  cfg1 / cfg2 / cfg2 with per-block parameter changes / cfg3 of BASELINE.json on one GPU (N = 1 only):
           ms per block, the kernel that ran, and the roofline fraction (HBM, or the FP32 issue rate for cfg3)
  strong   (N > 1) configs[4] read literally: the 65 536 streams SHARDED over the N GPUs, with and without the
           all-streams bus (fused per-tile sums + one pass + NCCL all-reduce) inside the timed region
  bus      the all-streams bus at full size (oalsfx_engine_mix_bus = mix + a deterministic reduction pass)
  e2e.link_peak   raw concurrent pinned H2D + D2H of the same bytes on the same box: the ceiling of the host-buffer path

  value  device-resident I/O (stream-major [stream][frame][channel] fp32 in HBM), CUDA events on the
         launching stream, max over ranks
  e2e    the same call with HOST buffers (pinned): H2D + kernel + D2H inside the timed region
  roofline      algorithmic HBM bytes (236 B/frame, SURVEY.md 8d / DESIGN.md) / event time of the
                fused kernel, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's own CPU implementation (oracle/_ref, compiled from the unmodified
                sources) on all host cores, bounded sample

`--impl reference` times that CPU implementation instead (bench.py's only other use of oracle/).
`--dump-outputs DIR` writes what the last timed step computed (rank 0) to DIR/output.npy (see dump_outputs), so that
two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STREAMS_PER_GPU = 65536
CHANNEL_FORMAT = 2  # stereo
CHANNELS = 2
RATE = 48000
BLOCK = 1024
CHAIN = (7, 1, 6, 11)  # equalizer, chorus, echo, eax_reverb (oalsfxpp::EffectType values)
BYTES_PER_FRAME = 236  # I/O 16 + reverb rings 192 + echo 12 + chorus 16 (SURVEY.md 8d)
CFG3_OPS_PER_FRAME = 266  # dry 2 + flanger 26 + ring modulator 60 + distortion 147 + compressor 31 (DESIGN.md section 5)
METRIC = "channel-samples/s, 4-slot EAX reverb chain @48 kHz"
UNIT = "channel-samples/s"
DUMP_BYTES = 32 << 20  # --dump-outputs: at most this much of the output (the cfg4 block is 512 MB)


def workload_config(streams):
    return {
        "workload": "cfg4: 4-slot chain equalizer+chorus+echo+eax_reverb (defaults), "
                    f"{streams} independent stereo 48 kHz streams per GPU, {BLOCK}-frame blocks",
        "streams_per_gpu": streams, "channels": CHANNELS, "rate": RATE, "block_frames": BLOCK,
        "layout": "stream-major [stream][frame][channel] fp32",
        "l2": "per-step working set (>10 GB of delay lines + 1 GB of I/O) exceeds the 126 MB L2; no flush needed",
        "parallelism": "streams sharded per GPU, no data-path collective",
    }


def dump_outputs(directory, np, torch, y):
    """Write y ([stream][frame][channel] fp32, what the caller of oalsfx_engine_mix receives) as DIR/output.npy: every
    stream when the block fits in DUMP_BYTES, else a fixed sample of streams (the same for every run with the same
    stream count), whose indices go to DIR/output_streams.npy (float64)."""
    streams = y.shape[0]
    keep = min(streams, DUMP_BYTES // (y[0].numel() * y.element_size()))
    index = np.arange(streams)
    if keep < streams:
        index = np.sort(np.random.default_rng(0).choice(streams, keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "output.npy"), y[torch.from_numpy(index).to(y.device)].cpu().numpy())
    np.save(os.path.join(directory, "output_streams.npy"), index.astype(np.float64))


# ---- CPU reference leg (test infrastructure under oracle/) ------------------------------------------
def _load_cpu_reference():
    """oracle/_ref (the compiled, unmodified reference) if present, else the restatement."""
    for kind, rel in (("reference", "oracle/_ref/liboalsfx_ref_fast.so"), ("reference", "oracle/_ref/liboalsfx_ref.so"),
                      ("port", "oracle/_build/liboalsfx_oracle.so")):
        path = os.path.join(ROOT, rel)
        if os.path.exists(path):
            lib = ctypes.CDLL(path)
            lib.orc_bench.argtypes = [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_int)] + [ctypes.c_int] * 3 + \
                [ctypes.c_uint32, ctypes.POINTER(ctypes.c_double)]
            lib.orc_bench.restype = ctypes.c_double
            return kind, lib
    return None, None  # build() makes oracle/_build; the tree is not written to from here


def cpu_run(lib, threads, streams, blocks):
    types = (ctypes.c_int * 4)(*CHAIN)
    checksum = ctypes.c_double()
    secs = lib.orc_bench(threads, streams, CHANNEL_FORMAT, RATE, types, 4, BLOCK, blocks, 0x0A15F00D,
                         ctypes.byref(checksum))
    return streams * CHANNELS * BLOCK * blocks / secs, secs


def cpu_baseline(target_seconds=12.0):
    kind, lib = _load_cpu_reference()
    if lib is None:
        return None
    threads = os.cpu_count() or 1
    per_stream_blocks = 64
    rate, _ = cpu_run(lib, threads, 2 * threads, per_stream_blocks)  # probe (same shape) to size the sample
    streams = max(threads, int(rate * target_seconds / (CHANNELS * BLOCK * per_stream_blocks)) // threads * threads)
    value, secs = cpu_run(lib, threads, streams, per_stream_blocks)
    return {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{streams} streams x {per_stream_blocks} blocks of {BLOCK} frames of the same 4-slot stereo chain, "
                      f"one Api instance per thread at a time, {secs:.1f} s wall"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    kind, lib = _load_cpu_reference()
    if lib is None:
        print(json.dumps({"impl": "reference", "unavailable": "no CPU checker library could be built"}))
        return 0
    threads = os.cpu_count() or 1
    blocks = 32
    rate, _ = cpu_run(lib, threads, 2 * threads, blocks)
    # each step: a bounded sample sized for ~2 s so K steps + W warm-ups stay within minutes
    streams = max(threads, int(rate * 2.0 / (CHANNELS * BLOCK * blocks)) // threads * threads)
    for _ in range(args.warmup):
        cpu_run(lib, threads, streams, blocks)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_run(lib, threads, streams, blocks)
    secs = time.perf_counter() - t0
    value = args.steps * streams * CHANNELS * BLOCK * blocks / secs
    sample = f"per step: {streams} streams x {blocks} blocks of {BLOCK} frames, {threads} threads"
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference", "config": workload_config(STREAMS_PER_GPU),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---- clocks ----------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled every few ms WHILE the timed region runs (NVML; falls back
    to the nvidia-smi query of B200_PROFILING.md when pynvml is unavailable)."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.sm, self.max_sm, self.reasons = index, [], None, set()
        self._stop, self._thread, self._nvml = threading.Event(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._handle, n.NVML_CLOCK_SM)))
        bits = n.nvmlDeviceGetCurrentClocksEventReasons(self._handle)
        for name, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
            if bits & getattr(n, attr, 0):
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [p.strip() for p in out.strip().split(",")]
        if len(parts) >= 6:
            self.sm.append(float(parts[0]))
            self.max_sm = float(parts[1])
            for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
                if parts[2 + i].lower().startswith("active"):
                    self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.004 if self._nvml else 0.1)

    def __enter__(self):
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no clock samples"]}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": "nvml" if self._nvml else "nvidia-smi"}


# ---- the other BASELINE.json configurations (one GPU, device buffers) --------------------------------
def secondary_configs(torch, ox, dev, stream, hbm_peak, sm_mhz):
    """cfg1, cfg2 (static and with per-block parameter changes), cfg3: median ms per 1024-frame block (CUDA events
    on the launching stream), the kernel the engine chose, and the roofline of each.  cfg3 is compute-bound: its
    roofline is the FP32 issue rate (148 SMs x 128 lanes x SM clock, one non-fused operation per lane and cycle --
    the path is compiled without FMA contraction) against 266 algorithmic operations per frame (DESIGN.md)."""
    import numpy as np
    T = ox.EffectType
    chain = [T.equalizer, T.chorus, T.echo, T.eax_reverb]

    def run(streams, fmt, rate, effects, schedule=None, blocks=24, warm=5):
        channels = ox.channel_count(fmt)
        x = torch.rand(streams, BLOCK, channels, device=dev) - 0.5
        y = torch.empty_like(x)
        host_s, times = 0.0, []
        with ox.Engine(streams, fmt, rate, len(effects), device=dev.index) as eng:
            for i, t in enumerate(effects):
                eng.set_effect(i, t)
            for b in range(warm + blocks):
                t0 = time.perf_counter()
                if schedule:
                    schedule(eng, b)
                t1 = time.perf_counter()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.mix(x, y, frames=BLOCK, stream=stream)
                e1.record()
                torch.cuda.synchronize()
                if b >= warm:
                    host_s += t1 - t0
                    times.append(e0.elapsed_time(e1))
            kernel = eng.last_kernel
        return float(np.median(times)), kernel, 1e3 * host_s / blocks, streams * BLOCK

    def cfg2_schedule(eng, b):  # a reverb gain ramp and an equalizer step every block, a tap change every 16 blocks
        rv = ox.default_props(T.eax_reverb, gain_=0.20 + 0.10 * ((b % 4) / 4.0), reflections_delay_=(0.012 if (b // 16) % 2 else 0.007))
        eq = ox.default_props(T.equalizer, mid1_gain_=1.0 + 0.5 * ((b % 8) / 8.0))
        eng.set_effect(3, T.eax_reverb, rv)
        eng.set_effect(0, T.equalizer, eq)

    def hbm(ms, frames, bytes_per_frame):
        achieved = bytes_per_frame * frames / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "algorithmic_bytes_per_frame": bytes_per_frame}

    out = {}
    ms, k, _, fr = run(1024, ox.ChannelFormat.mono, 48000, [T.eax_reverb])
    out["cfg1"] = {"workload": "EAX reverb (default preset), 1024 mono 48 kHz streams", "ms_per_block": ms, "kernel": k,
                   "roofline": hbm(ms, fr, 200)}
    ms, k, _, fr = run(4096, ox.ChannelFormat.stereo, 48000, chain)
    out["cfg2"] = {"workload": "equalizer+chorus+echo+EAX reverb, 4096 stereo 48 kHz streams, static parameters",
                   "ms_per_block": ms, "kernel": k, "roofline": hbm(ms, fr, BYTES_PER_FRAME)}
    ms, k, host_ms, fr = run(4096, ox.ChannelFormat.stereo, 48000, chain, schedule=cfg2_schedule, blocks=48)
    out["cfg2_ramps"] = {"workload": "the same with parameter changes before every block (reverb gain ramp, equalizer step; reflections delay every 16 blocks)",
                         "ms_per_block": ms, "kernel": k, "host_param_update_ms_per_block": host_ms, "roofline": hbm(ms, fr, BYTES_PER_FRAME)}
    ms, k, _, fr = run(16384, ox.ChannelFormat.mono, 96000, [T.flanger, T.ring_modulator, T.distortion, T.compressor])
    fp32_peak = 148 * 128 * (sm_mhz or 1965.0) * 1e6 / 1e12
    achieved = CFG3_OPS_PER_FRAME * fr / (ms * 1e-3) / 1e12
    out["cfg3"] = {"workload": "flanger+ring modulator+distortion+compressor, 16384 mono 96 kHz streams", "ms_per_block": ms, "kernel": k,
                   "roofline": {"bound": "fp32_issue", "achieved": achieved, "peak": fp32_peak, "unit": "Tflop/s (non-fused FP32 operations)",
                                "frac": achieved / fp32_peak, "algorithmic_ops_per_frame": CFG3_OPS_PER_FRAME,
                                "hbm_GBps": 24 * fr / (ms * 1e-3) / 1e9}}
    return out


def link_peak(torch, dev, nbytes, world, dist):
    """Raw pinned-memory copies of the e2e path's bytes, both directions at once on two streams (what a perfect
    overlap of the host-buffer path could reach on this box)."""
    h_in = torch.empty(nbytes // 4, dtype=torch.float32).pin_memory()
    h_out = torch.empty(nbytes // 4, dtype=torch.float32).pin_memory()
    d_in = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    d_out = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    reps = 4

    def once():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)

    once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    torch.cuda.synchronize()
    secs = (time.perf_counter() - t0) / reps
    t = torch.tensor([secs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t.item())
    return {"seconds_per_step_of_copies": secs, "h2d_plus_d2h_GBps_per_gpu": 2 * nbytes / secs / 1e9,
            "what": f"{nbytes >> 20} MiB pinned H2D and {nbytes >> 20} MiB D2H concurrently on two streams, every rank at once, max over ranks"}


# ---- our arm ---------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU, help="streams per GPU (default: the cfg4 size)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="leave out the cfg1 / cfg2 / cfg3 records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step (a fixed sample of at most 32 MB of it) to DIR/output.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import oalsfxpp_b200 as ox

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Rank 0 prints ONE JSON line on stdout and nothing else: anything a library writes to file descriptor 1
    # (NCCL's version banner does, whatever NCCL_DEBUG says) is sent to stderr instead.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    S, C, F = args.streams, CHANNELS, BLOCK

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = ox.Engine(S, CHANNEL_FORMAT, RATE, 4, device=local_rank)
    for slot, fx in enumerate(CHAIN):
        eng.set_effect(slot, fx)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x0A15F00D + rank)
    x = torch.rand((S, F, C), device=dev, generator=gen, dtype=torch.float32) - 0.5  # white noise in [-0.5, 0.5)
    y = torch.empty_like(x)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        eng.mix(x, y, frames=F, stream=stream)

    # -- device-resident throughput ---------------------------------------------------------------------
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = eng.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with ClockSampler(local_rank) as clocks:
        ev[0].record()
        for k in range(args.steps):
            step_device()
            ev[k + 1].record()
        barrier()
    launches = eng.launch_count - launches0
    device_bytes = eng.device_bytes
    headline_kernel = eng.last_kernel  # the kernel the timed launches actually were (oalsfx_engine_last_kernel)
    total_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = sorted(ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps))
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * S * C * F * args.steps / (total_ms_max * 1e-3)
    assert bool(torch.isfinite(y).all()), "non-finite output"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np, torch, y)  # before the legs below overwrite y

    # -- the all-streams output bus (BASELINE config 4) at full size: oalsfx_engine_mix_bus = mix + one deterministic pass
    #    over the block's output + (N > 1) one NCCL all-reduce of the [frames][channels] bus over NVLink.
    #    `extra_ms_per_block` = what the bus costs on top of the plain mix.
    bus = torch.zeros((F, C), device=dev, dtype=torch.float32)
    bus_steps = max(3, min(args.steps, 10))

    def step_bus():
        eng.mix_bus(x, y, F, bus, stream=stream)
        if world > 1:
            dist.all_reduce(bus, op=dist.ReduceOp.SUM)

    step_bus()
    barrier()
    bus_kernel = eng.last_kernel
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    for _ in range(bus_steps):
        step_bus()
    b1.record()
    barrier()
    t = torch.tensor([b0.elapsed_time(b1) / bus_steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    bus_ms = float(t.item())
    # the reduction pass alone (events around it; the subtraction above is between two timed regions and noisy)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for _ in range(bus_steps):
        eng.reduce_bus(F, y, bus, stream=stream)
    r1.record()
    torch.cuda.synchronize()
    reduce_ms = r0.elapsed_time(r1) / bus_steps
    bus_check = float((bus.double() - (y.double().sum(dim=0) if world == 1 else bus.double())).abs().max().item())
    bus_info = {"ms_per_block_mix_plus_bus": bus_ms, "extra_ms_per_block": bus_ms - total_ms_max / args.steps,
                "reduce_pass_ms_per_block": reduce_ms, "kernel": bus_kernel,
                "what": "oalsfx_engine_mix_bus: mix + oalsfx_engine_reduce_bus (two coalesced passes over the block's output) on one stream" +
                        (f" + NCCL all_reduce of [{F}][{C}] fp32 over {world} GPUs" if world > 1 else ""),
                "bytes_read_for_the_bus_per_gpu": S * F * C * 4,
                "max_abs_diff_vs_float64_sum_of_rows": bus_check if world == 1 else None}

    # -- end to end through the C ABI with host buffers ---------------------------------------------------
    e2e = None
    if not args.skip_e2e:
        hx = torch.empty((S, F, C), dtype=torch.float32).pin_memory()
        hx.copy_(x.cpu())
        hy = torch.empty((S, F, C), dtype=torch.float32).pin_memory()
        hxn, hyn = hx.numpy(), hy.numpy()
        e2e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            eng.mix(hxn, hyn, frames=F)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.mix(hxn, hyn, frames=F)  # H2D + fused kernel + D2H + sync inside the call
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": world * S * C * F * e2e_steps / float(t.item()), "unit": UNIT,
               "h2d_bytes_per_step": S * F * C * 4, "d2h_bytes_per_step": S * F * C * 4, "steps": e2e_steps,
               "note": "oalsfx_engine_mix with pinned host buffers: H2D + kernel + D2H inside the timed region"}
        # the same call with the caller's buffers as an unmodified host program would have them (pageable, from the C
        # allocator), and after oalsfx_engine_pin_host has page-locked them in place
        def e2e_rate(a_in, a_out, steps):
            eng.mix(a_in, a_out, frames=F)
            barrier()
            t_0 = time.perf_counter()
            for _ in range(steps):
                eng.mix(a_in, a_out, frames=F)
            barrier()
            tt = torch.tensor([time.perf_counter() - t_0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return world * S * C * F * steps / float(tt.item())

        px = np.array(hxn, copy=True)
        py = np.empty_like(px)
        e2e["pageable_buffers"] = {"value": e2e_rate(px, py, 3), "unit": UNIT}
        eng.pin_host(px)
        eng.pin_host(py)
        e2e["pageable_buffers_after_pin_host"] = {"value": e2e_rate(px, py, 5), "unit": UNIT,
                                                  "note": "oalsfx_engine_pin_host (cudaHostRegister in place); OALSFX_PIN_HOST=1 does it on first sight"}
        eng.unpin_host(px)
        eng.unpin_host(py)
        del hx, hy, hxn, hyn, px, py
        lp = link_peak(torch, dev, S * F * C * 4, world, dist if world > 1 else None)
        lp["channel_samples_per_s_if_copies_were_all"] = world * S * C * F / lp["seconds_per_step_of_copies"]
        e2e["link_peak"] = lp
        e2e["fraction_of_link_peak"] = e2e["value"] / lp["channel_samples_per_s_if_copies_were_all"]

    # -- strong scaling: BASELINE configs[4] read literally -- the 65 536 streams sharded over the N GPUs ------
    strong = None
    if world > 1:
        eng.close()
        del x, y
        torch.cuda.empty_cache()
        Ss = STREAMS_PER_GPU // world
        eng = ox.Engine(Ss, CHANNEL_FORMAT, RATE, 4, device=local_rank)
        for slot, fx in enumerate(CHAIN):
            eng.set_effect(slot, fx)
        x = torch.rand((Ss, F, C), device=dev, generator=gen, dtype=torch.float32) - 0.5
        y = torch.empty_like(x)

        def timed(fn):
            for _ in range(args.warmup):
                fn()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            barrier()
            tt = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        def strong_step():
            eng.mix(x, y, frames=F, stream=stream)

        def strong_step_bus():
            eng.mix_bus(x, y, F, bus, stream=stream)
            dist.all_reduce(bus, op=dist.ReduceOp.SUM)

        ms_plain = timed(strong_step)
        k_plain = eng.last_kernel
        ms_bus = timed(strong_step_bus)
        k_bus = eng.last_kernel
        strong = {"streams_total": Ss * world, "streams_per_gpu": Ss, "ms_per_step": ms_plain, "kernel": k_plain,
                  "value": Ss * world * C * F / (ms_plain * 1e-3), "unit": UNIT,
                  "with_bus_in_timed_region": {"ms_per_step": ms_bus, "kernel": k_bus, "value": Ss * world * C * F / (ms_bus * 1e-3),
                                               "what": "mix + per-GPU bus (oalsfx_engine_mix_bus) + NCCL all_reduce of the [frames][channels] bus, all inside the timed region"},
                  "one_gpu_same_streams": {"value": value / world, "unit": UNIT,
                                           "what": "this run's weak leg: %d streams on ONE GPU (max over ranks)" % S}}
        strong["speedup_over_one_gpu"] = strong["value"] / strong["one_gpu_same_streams"]["value"]
        strong["speedup_over_one_gpu_with_bus"] = strong["with_bus_in_timed_region"]["value"] / strong["one_gpu_same_streams"]["value"]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    median_ms = kernel_ms[len(kernel_ms) // 2]
    achieved = BYTES_PER_FRAME * S * F / (median_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_path):
        tj = json.load(open(traffic_path))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    clock_summary = clocks.summary()
    configs = None
    if world == 1 and not args.skip_configs:
        eng.close()
        del x, y
        torch.cuda.empty_cache()
        configs = secondary_configs(torch, ox, dev, stream, peak, clock_summary.get("sm_mhz"))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (uniform white noise in [-0.5, 0.5) from torch.rand -- not the hash noise of the parity tests)",
        "config": workload_config(S),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": f"{headline_kernel} (reported by the engine after the timed launches; kDuoChainStereo = "
                               "duo_kernel<2,FxEqualizer,FxModDelay,FxEcho,FxReverb>): one launch = one step = the whole fused path",
                     "algorithmic_bytes_per_launch": BYTES_PER_FRAME * S * F, "kernel_ms_median": median_ms,
                     "peak_source": peak_src},
        "clocks": clock_summary,
        "gpu_launches": launches,
        "bus": bus_info,
        "device_bytes": device_bytes,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if strong is not None:
        line["strong"] = strong
    if configs is not None:
        line["configs"] = configs
    if world == 1 and not args.skip_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

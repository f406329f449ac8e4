#!/usr/bin/env python3
"""Bus formats and pan routes (oalsfx_engine_set_bus_format / set_route_pans): ms per reduce_buses call on 65 536 streams x
1024-frame blocks.

The block `dst` is seeded once in device memory (256-768 MB, above the 126 MB L2); every case is the median of CUDA-event
pairs around 60 calls on the launching stream after 5 warm-up calls (route_timing.py's method).  No mix runs between the
calls, so the frame clock stands still and a ramping plan stays ramping for every timed call.  One route per stream, K = 64
contiguous buses (tile-aligned runs) unless noted:

  * mono -> stereo steady pans against the mono and stereo unweighted reductions (route_streams at the engine's format);
  * stereo -> stereo with a full 2x2 matrix and stereo -> 5.1, steady, against one steady scalar route per stream;
  * every pan case ramping, against the same plan steady;
  * TILED with 4096 random send buses (record only);
  * host wall time of a coefficient-only set_route_pans on all streams plus the next reduce_buses, synchronized;
  * route_timing.py rerun in the same call (its record under "route_timing_rerun") and, with --bench, bench.py's line.

    python profiles/pan_timing.py --bench --out profiles/r03_pan_timing.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oalsfxpp_b200 as ox  # noqa: E402
from oalsfxpp_b200 import ChannelFormat as F  # noqa: E402

S, FRAMES = 65536, 1024
CALLS, WARM = 60, 5
LAYOUTS = (("stream_major", ox.LAYOUT_STREAM_MAJOR), ("tiled", ox.LAYOUT_TILED))


def median_ms(fn, calls=CALLS, warm=WARM):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def to_tiled(x):
    C = x.shape[2]
    return x.reshape(S // 32, 32, FRAMES, C).permute(0, 2, 3, 1).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_pan_timing.json"))
    ap.add_argument("--bench", action="store_true", help="also run bench.py --gpus 1 --steps 20 --warmup 5 and keep its line")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    stream = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(1)
    contiguous = (np.arange(S, dtype=np.int64) * 64 // S).astype(np.int32)
    random = (64 + rng.integers(0, 4096, S)).astype(np.int32)
    n_buses = 64 + 4096
    rows = []

    def timed(eng, bufs, case, **extra):
        buses = torch.empty(n_buses, FRAMES, eng.bus_channels, device=dev)
        rec = {"case": case, **extra}
        for name, layout in LAYOUTS:
            rec[f"{name}_ms"] = median_ms(lambda: eng.reduce_buses(FRAMES, bufs[name], buses, layout=layout, stream=stream))
        rows.append(rec)
        return rec

    def ratio(rec, base, what):
        for name, _ in LAYOUTS:
            rec[f"{name}_over_{what}"] = rec[f"{name}_ms"] / base[f"{name}_ms"]

    unweighted, steady_one = {}, None
    for fmt in (F.mono, F.stereo):
        C = ox.channel_count(fmt)
        gen = torch.Generator(device=dev).manual_seed(3)
        y = torch.rand(S, FRAMES, C, device=dev, generator=gen) - 0.5
        bufs = {"stream_major": y, "tiled": to_tiled(y)}
        with ox.Engine(S, fmt, 48000, 1) as eng:
            eng.route(contiguous)
            unweighted[fmt] = timed(eng, bufs, "route_streams", fmt=fmt.name, routing="64_contiguous")
            if fmt == F.stereo:
                eng.set_routes(contiguous[:, None], (0.25 + rng.random((S, 1))).astype(np.float32))
                steady_one = timed(eng, bufs, "one_route_steady_gain", fmt="stereo", routing="64_contiguous")
            pairs = [(F.stereo, "64_contiguous", contiguous)] if fmt == F.mono else \
                [(F.stereo, "64_contiguous", contiguous), (F.five_point_one, "64_contiguous", contiguous)]
            if fmt == F.mono:
                pairs.append((F.stereo, "4096_random", random))
            for bus_fmt, kind, routing in pairs:
                eng.set_routes(routing[:, None], np.ones((S, 1), np.float32))
                eng.set_bus_format(bus_fmt)
                Cb = ox.channel_count(bus_fmt)
                pan = (0.25 + rng.random((S, Cb, C))).astype(np.float32)
                eng.set_route_pans(pan, routing)
                label = f"{fmt.name}_to_{bus_fmt.name}"
                steady = timed(eng, bufs, "pan_steady", pair=label, routing=kind)
                eng.set_route_pans(pan * np.float32(0.5), routing, ramp_frames=1 << 24)
                ramp = timed(eng, bufs, "pan_ramping", pair=label, routing=kind)
                ratio(ramp, steady, "steady")
                if fmt == F.mono and kind == "64_contiguous":
                    ratio(steady, unweighted[F.mono], "mono_unweighted")
                elif fmt == F.stereo:
                    ratio(steady, steady_one, "one_route_steady_gain")
                steady["tiled_over_stream_major"] = steady["tiled_ms"] / steady["stream_major_ms"]
                if kind == "64_contiguous" and (fmt == F.mono or bus_fmt == F.five_point_one):
                    # coefficient-only change on every stream + the next reduce, host wall time to the end of the device work
                    buses = torch.empty(n_buses, FRAMES, Cb, device=dev)
                    eng.set_route_pans(pan, routing)
                    eng.reduce_buses(FRAMES, y, buses, stream=stream)
                    torch.cuda.synchronize()
                    walls, alone = [], []
                    for i in range(20):
                        m = pan * np.float32(1.0 + 0.01 * (i % 2))
                        t0 = time.perf_counter()
                        eng.set_route_pans(m, routing)
                        eng.reduce_buses(FRAMES, y, buses, stream=stream)
                        torch.cuda.synchronize()
                        walls.append((time.perf_counter() - t0) * 1e3)
                        t0 = time.perf_counter()
                        eng.reduce_buses(FRAMES, y, buses, stream=stream)
                        torch.cuda.synchronize()
                        alone.append((time.perf_counter() - t0) * 1e3)
                    rows.append({"case": "coefficient_only_set_route_pans_plus_reduce_wall", "pair": label,
                                 "median_ms": float(np.median(walls)), "reduce_alone_wall_median_ms": float(np.median(alone)),
                                 "device_bytes": eng.device_bytes})
                eng.route(contiguous)                       # scalar routes again: the next format change is allowed
                eng.set_bus_format(fmt)
        del y, bufs
        torch.cuda.empty_cache()

    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_clock_max_clock": smi[0] if smi else "",
              "streams": S, "block_frames": FRAMES, "calls_per_median": CALLS, "cases": rows}
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "route_timing.json")
        subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "route_timing.py"), "--out", out], check=True,
                       stdout=subprocess.DEVNULL)
        with open(out) as f:
            result["route_timing_rerun"] = json.load(f)
    if args.bench:
        line = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "20", "--warmup", "5"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
        result["bench"] = json.loads(line)
    text = json.dumps(result, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()

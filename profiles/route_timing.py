#!/usr/bin/env python3
"""Routes with gains (oalsfx_engine_set_routes): ms per reduce_buses call on 65 536 stereo streams x 1024-frame blocks.

The block `dst` is seeded once in device memory (512 MB, above the 126 MB L2); every case is the median of CUDA-event
pairs around 60 calls on the launching stream after 5 warm-up calls (bus_timing.py's method).  No mix runs between the
calls, so the frame clock stands still and a ramping plan stays ramping for every timed call.

  * unity: set_routes with gain 1 against route_streams on the same routing (both run the unweighted kernels);
  * steady: one route per stream with non-unity gains, K = 64 contiguous and 4096 random buses, against unweighted
    reduce_buses on the same routing;
  * two routes per stream: 64 category buses + 4096 random send buses, steady gains, against the one-route cases;
  * ramping: the one-route and two-route plans with a ramp covering the block, against the same plans steady;
  * host wall time of a gain-only set_routes on all streams plus the next reduce_buses, synchronized (time.perf_counter).

    python profiles/route_timing.py --out profiles/r03_route_timing.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oalsfxpp_b200 as ox  # noqa: E402
from oalsfxpp_b200 import ChannelFormat as F  # noqa: E402

S, FRAMES, C = 65536, 1024, 2
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
    return x.reshape(S // 32, 32, FRAMES, C).permute(0, 2, 3, 1).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_route_timing.json"))
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    stream = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(3)
    y = torch.rand(S, FRAMES, C, device=dev, generator=gen) - 0.5
    bufs = {"stream_major": y, "tiled": to_tiled(y)}
    rng = np.random.default_rng(1)
    contiguous = (np.arange(S, dtype=np.int64) * 64 // S).astype(np.int32)
    random = (64 + rng.integers(0, 4096, S)).astype(np.int32)
    n_buses = 64 + 4096
    gains1 = (0.25 + rng.random((S, 1))).astype(np.float32)
    gains2 = (0.25 + rng.random((S, 2))).astype(np.float32)
    buses = torch.empty(n_buses, FRAMES, C, device=dev)
    rows = []

    def timed(eng, case, **extra):
        rec = {"case": case, **extra}
        for name, layout in LAYOUTS:
            rec[f"{name}_ms"] = median_ms(lambda: eng.reduce_buses(FRAMES, bufs[name], buses, layout=layout, stream=stream))
        rows.append(rec)
        return rec

    with ox.Engine(S, F.stereo, 48000, 1) as eng:
        one = {}
        for kind, routing in (("64_contiguous", contiguous), ("4096_random", random)):
            eng.route(routing)
            base = timed(eng, "route_streams", routing=kind)
            eng.set_routes(routing[:, None], np.ones((S, 1), np.float32))
            unity = timed(eng, "set_routes_unity", routing=kind)
            eng.set_routes(routing[:, None], gains1)
            steady = timed(eng, "one_route_steady", routing=kind)
            eng.set_routes(routing[:, None], gains1 * 0.5, ramp_frames=1 << 24)
            ramp = timed(eng, "one_route_ramping", routing=kind)
            one[kind] = steady
            for name, _ in LAYOUTS:
                unity[f"{name}_over_route_streams"] = unity[f"{name}_ms"] / base[f"{name}_ms"]
                steady[f"{name}_over_unweighted"] = steady[f"{name}_ms"] / base[f"{name}_ms"]
                ramp[f"{name}_over_steady"] = ramp[f"{name}_ms"] / steady[f"{name}_ms"]
        both = np.stack([contiguous, random], axis=1)
        eng.set_routes(both, gains2)
        two = timed(eng, "two_routes_steady", routing="64_contiguous+4096_random")
        eng.set_routes(both, gains2 * 0.5, ramp_frames=1 << 24)
        two_ramp = timed(eng, "two_routes_ramping", routing="64_contiguous+4096_random")
        for name, _ in LAYOUTS:
            for kind in one:
                two[f"{name}_over_one_route_{kind}"] = two[f"{name}_ms"] / one[kind][f"{name}_ms"]
            two_ramp[f"{name}_over_steady"] = two_ramp[f"{name}_ms"] / two[f"{name}_ms"]

        # gain-only change on every stream + the next reduce, host wall time to the end of the device work
        for routes, (b, g_base) in ((1, (random[:, None], gains1)), (2, (both, gains2))):
            eng.set_routes(b, g_base)
            eng.reduce_buses(FRAMES, y, buses, stream=stream)
            torch.cuda.synchronize()
            walls, alone = [], []
            for i in range(20):
                g = g_base * np.float32(1.0 + 0.01 * (i % 2))
                t0 = time.perf_counter()
                eng.set_routes(b, g)
                eng.reduce_buses(FRAMES, y, buses, stream=stream)
                torch.cuda.synchronize()
                walls.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                eng.reduce_buses(FRAMES, y, buses, stream=stream)
                torch.cuda.synchronize()
                alone.append((time.perf_counter() - t0) * 1e3)
            rows.append({"case": "gain_only_set_routes_plus_reduce_wall", "routes_per_stream": routes,
                         "median_ms": float(np.median(walls)), "reduce_alone_wall_median_ms": float(np.median(alone)),
                         "device_bytes": eng.device_bytes})

    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_clock_max_clock": smi[0] if smi else "",
              "streams": S, "block_frames": FRAMES, "channels": C, "calls_per_median": CALLS, "cases": rows}
    text = json.dumps(result, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Submix buses (oalsfx_engine_reduce_buses / mix_buses): ms per call on 65 536 stereo streams x 1024-frame blocks.

The block `dst` is seeded once in device memory (512 MB, above the 126 MB L2) and every case is the median of CUDA-event
pairs around 60 calls on the launching stream after 5 warm-up calls:

  * reduce_buses, K in {1, 64, 4096, 65536} buses x {contiguous routing (bus = s * K / S: whole tiles for K <= 2048),
    random routing} x {STREAM_MAJOR, TILED};
  * reduce_bus (the all-streams bus), for reference;
  * torch index_add_ over [S][frames * C] rows (what a host does without the engine; atomics, not deterministic);
  * mix_buses against mix on the cfg4 chain (equalizer + chorus + echo + EAX reverb), K = 64 contiguous and 4096 random.

Bytes per call = member rows read + partial rows written and read + bus rows written; `of_copy_bw` is that over the time,
as a fraction of the 6.55 TB/s device-to-device copy rate DESIGN.md reports against.

    python profiles/bus_timing.py > profiles/r03_bus_timing.json
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oalsfxpp_b200 as ox  # noqa: E402
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T  # noqa: E402

S, FRAMES, C = 65536, 1024, 2
COPY_BW = 6.55e12
CHAIN = [T.equalizer, T.chorus, T.echo, T.eax_reverb]
CALLS, WARM = 60, 5


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


def plan_bytes(routing, n_buses):
    """Bytes one reduce_buses call moves: member rows, partial rows (written once, read once), bus rows."""
    row = FRAMES * C * 4
    counts = np.bincount(routing[routing >= 0], minlength=n_buses)
    partial_rows = 0
    lens = counts[counts > 32]
    while lens.size:
        runs = -(-lens // 32)
        partial_rows += int(runs.sum())
        lens = runs[runs > 32]
    return int(counts.sum()) * row + 2 * partial_rows * row + n_buses * row


def routings():
    rng = np.random.default_rng(1)
    out = []
    for k in (1, 64, 4096, 65536):
        out.append((k, "contiguous", (np.arange(S, dtype=np.int64) * k // S).astype(np.int32)))
        if k > 1:
            out.append((k, "random", rng.integers(0, k, S).astype(np.int32)))
    return out


def to_tiled(x):
    return x.reshape(S // 32, 32, FRAMES, C).permute(0, 2, 3, 1).contiguous()


def reduce_cases(stream):
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(3)
    y = torch.rand(S, FRAMES, C, device=dev, generator=gen) - 0.5
    yt = to_tiled(y)
    rows = []
    with ox.Engine(S, F.stereo, 48000, 1) as eng:
        bus = torch.empty(FRAMES, C, device=dev)
        ref = {}
        for name, layout, buf in (("stream_major", ox.LAYOUT_STREAM_MAJOR, y), ("tiled", ox.LAYOUT_TILED, yt)):
            ref[name] = median_ms(lambda: eng.reduce_bus(FRAMES, buf, bus, layout=layout, stream=stream))
        rows.append({"case": "reduce_bus", "stream_major_ms": ref["stream_major"], "tiled_ms": ref["tiled"],
                     "bytes": S * FRAMES * C * 4 + FRAMES * C * 4})
        for k, kind, routing in routings():
            eng.route(routing)
            buses = torch.empty(k, FRAMES, C, device=dev)
            rec = {"case": "reduce_buses", "buses": k, "routing": kind, "bytes": plan_bytes(routing, k)}
            for name, layout, buf in (("stream_major", ox.LAYOUT_STREAM_MAJOR, y), ("tiled", ox.LAYOUT_TILED, yt)):
                before = eng.launch_count
                eng.reduce_buses(FRAMES, buf, buses, layout=layout, stream=stream)
                rec["launches"] = eng.launch_count - before
                ms = median_ms(lambda: eng.reduce_buses(FRAMES, buf, buses, layout=layout, stream=stream))
                rec[f"{name}_ms"] = ms
                rec[f"{name}_over_reduce_bus"] = ms / ref[name]
                rec[f"{name}_of_copy_bw"] = rec["bytes"] / (ms * 1e-3) / COPY_BW
            index = torch.from_numpy(routing.astype(np.int64)).to(dev)
            flat = y.view(S, FRAMES * C)
            out = torch.empty(k, FRAMES * C, device=dev)
            rec["torch_index_add_ms"] = median_ms(lambda: out.zero_().index_add_(0, index, flat))
            rows.append(rec)
    return rows


def mix_cases(stream):
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(4)
    x = torch.rand(S, FRAMES, C, device=dev, generator=gen) - 0.5
    y = torch.empty_like(x)
    rng = np.random.default_rng(2)
    rows = []
    with ox.Engine(S, F.stereo, 48000, 4) as eng:
        for i, t in enumerate(CHAIN):
            eng.set_effect(i, t)
        for k, kind, routing in ((64, "contiguous", ((np.arange(S) * 64) // S).astype(np.int32)),
                                 (4096, "random", rng.integers(0, 4096, S).astype(np.int32))):
            eng.route(routing)
            buses = torch.empty(k, FRAMES, C, device=dev)
            mix_ms = median_ms(lambda: eng.mix(x, y, frames=FRAMES, stream=stream), calls=30)
            both_ms = median_ms(lambda: eng.mix_buses(x, y, FRAMES, buses, stream=stream), calls=30)
            alone_ms = median_ms(lambda: eng.reduce_buses(FRAMES, y, buses, stream=stream))
            rows.append({"case": "mix_buses_cfg4", "buses": k, "routing": kind, "mix_ms": mix_ms, "mix_buses_ms": both_ms,
                         "difference_ms": both_ms - mix_ms, "reduce_buses_alone_ms": alone_ms, "kernel": eng.last_kernel})
    return rows


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    stream = torch.cuda.current_stream().cuda_stream
    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_clock_max_clock": smi[0] if smi else "",
              "streams": S, "block_frames": FRAMES, "channels": C, "calls_per_median": CALLS,
              "reduce": reduce_cases(stream), "mix": mix_cases(stream)}
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Stream placement inside the engine (OALSFX_PLACEMENT_AUTO): ms per 1024-frame block of the cfg4 chain with 113 reverb
presets assigned as stream s -> preset s mod 113, device-resident buffers in the caller's order, CUDA events on the
launching stream (medians), for

  * table mode: CALLER placement, the presets left in the caller's order;
  * AUTO placement, steady state (class-per-tile launch plus the two I/O permutation passes);
  * the caller-ordered engine of oalsfx_plan_placement (the host reorders its buffers once);
  * the first AUTO block: every stream moves (host wall clock, planning + lane moves + the block);
  * the block after 64 scattered streams change preset, and the one after it (host wall clock).

    python profiles/placement_timing.py > profiles/r03_placement_timing.json
"""
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
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T  # noqa: E402

BLOCK = 1024
CHAIN = [T.equalizer, T.chorus, T.echo]


def configure(eng, preset_of_stream, props):
    for i, t in enumerate(CHAIN):
        eng.set_effect(i, t)
    s, n = 0, len(preset_of_stream)
    while s < n:  # one call per run of equal presets
        e = s + 1
        while e < n and preset_of_stream[e] == preset_of_stream[s]:
            e += 1
        eng.set_effect(3, T.eax_reverb, props[preset_of_stream[s]], first_stream=s, n_streams=e - s)
        s = e


def timed_block(eng, x, y, stream):
    """(device ms by events, host wall ms incl. synchronize) of one block."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    eng.mix(x, y, frames=BLOCK, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3


def steady(eng, x, y, stream, blocks=12, warm=3):
    for _ in range(warm):
        timed_block(eng, x, y, stream)
    return float(np.median([timed_block(eng, x, y, stream)[0] for _ in range(blocks)]))


def measure(n):
    props = [ox.reverb_preset(g, m) for g, m in ox.reverb_preset_names()]
    presets = [s % len(props) for s in range(n)]
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(n)
    x = torch.rand(n, BLOCK, 2, device=dev, generator=gen) - 0.5
    y = torch.empty_like(x)
    stream = torch.cuda.current_stream().cuda_stream
    out = {"streams": n, "presets": len(props)}
    with ox.Engine(n, F.stereo, 48000, 4) as eng:
        configure(eng, presets, props)
        out["table_mode_ms"] = steady(eng, x, y, stream)
        out["table_mode_kernel"] = eng.last_kernel
    with ox.Engine(n, F.stereo, 48000, 4) as eng:
        configure(eng, presets, props)
        eng.set_placement("auto")
        dev_ms, wall_ms = timed_block(eng, x, y, stream)
        out["auto_first_block_wall_ms"] = wall_ms
        out["auto_first_block_device_ms"] = dev_ms
        timed_block(eng, x, y, stream)  # the block after the update bits were consumed
        before = eng.launch_count
        out["auto_steady_ms"] = steady(eng, x, y, stream)
        out["auto_launches_per_block"] = (eng.launch_count - before) / 15
        out["auto_kernel"] = eng.last_kernel
        out["auto_lanes"] = eng.lanes()[1]
        out["auto_device_bytes"] = eng.device_bytes
        rng = np.random.default_rng(64)
        changed = rng.choice(n, 64, replace=False)
        lanes_before = eng.lane_of_stream
        for s in changed:
            eng.set_effect(3, T.eax_reverb, props[(presets[s] + 1 + int(s) % 7) % len(props)], first_stream=int(s), n_streams=1)
        dev_ms, wall_ms = timed_block(eng, x, y, stream)
        out["after_64_changes_wall_ms"] = wall_ms
        out["after_64_changes_device_ms"] = dev_ms
        out["after_64_changes_streams_moved"] = int((eng.lane_of_stream != lanes_before).sum())
        dev_ms, wall_ms = timed_block(eng, x, y, stream)
        out["second_block_after_changes_wall_ms"] = wall_ms
        out["second_block_after_changes_device_ms"] = dev_ms
        out["auto_steady_after_changes_ms"] = steady(eng, x, y, stream, blocks=6, warm=1)
    index, total, classes = ox.plan_placement(np.array(presets, dtype=np.int32))
    ordered = [0] * total
    for label, first, span in classes:
        ordered[first:first + span] = [label] * span
    xo = torch.zeros(total, BLOCK, 2, device=dev)
    xo[torch.from_numpy(index.astype(np.int64)).to(dev)] = x
    yo = torch.empty_like(xo)
    with ox.Engine(total, F.stereo, 48000, 4) as eng:
        configure(eng, ordered, props)
        out["caller_ordered_ms"] = steady(eng, xo, yo, stream)
        out["caller_ordered_streams"] = total
        out["caller_ordered_kernel"] = eng.last_kernel
    return out


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "", "block_frames": BLOCK,
              "chain": "equalizer+chorus+echo+eax_reverb, slot 3 preset s mod 113", "runs": [measure(n) for n in (16384, 65536)]}
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()

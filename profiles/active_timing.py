#!/usr/bin/env python3
"""Paused streams (oalsfx_engine_set_active): ms per 1024-frame block of the cfg4 chain, device-resident buffers in the
caller's order, CUDA events on the launching stream (medians), for

  * AUTO placement: 65 536 streams with 113 reverb presets as stream s -> preset s mod 113, 100 / 50 / 25 / 10 % of them
    active (a random set, fixed per fraction), each next to an AUTO engine that holds only the active streams with the
    same presets;
  * CALLER placement: one preset, 65 536 streams with 3 of every 4 tiles paused, next to a 16 384-stream engine;
  * churn: in the 25 % engine, the block after 64 scattered streams pause and 64 others resume, and the block after it
    (host wall clock, as profiles/placement_timing.py).

    python profiles/active_timing.py > profiles/r03_active_timing.json
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
STREAMS = 65536


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


def set_active(eng, active):
    """Pause every stream outside `active` (one call per run)."""
    s, n = 0, len(active)
    while s < n:
        e = s + 1
        while e < n and active[e] == active[s]:
            e += 1
        if not active[s]:
            eng.set_active(False, s, e - s)
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
    before = eng.launch_count
    ms = float(np.median([timed_block(eng, x, y, stream)[0] for _ in range(blocks)]))
    return ms, (eng.launch_count - before) / blocks, eng.last_kernel


def auto_runs(x, y, stream):
    props = [ox.reverb_preset(g, m) for g, m in ox.reverb_preset_names()]
    presets = [s % len(props) for s in range(STREAMS)]
    runs = []
    for fraction in (1.0, 0.5, 0.25, 0.10):
        rng = np.random.default_rng(int(fraction * 1000))
        n_active = int(round(STREAMS * fraction))
        active = np.zeros(STREAMS, dtype=bool)
        active[rng.choice(STREAMS, n_active, replace=False)] = True
        out = {"active_fraction": fraction, "active_streams": n_active}
        with ox.Engine(STREAMS, F.stereo, 48000, 4) as eng:
            configure(eng, presets, props)
            eng.set_placement("auto")
            set_active(eng, active)
            out["auto_ms"], out["auto_launches_per_block"], out["auto_kernel"] = steady(eng, x, y, stream)
            out["auto_lanes"] = eng.lanes()[1]
            if fraction == 0.25:
                churn = {}
                off = rng.choice(np.flatnonzero(active), 64, replace=False)
                on = rng.choice(np.flatnonzero(~active), 64, replace=False)
                lanes_before = eng.lane_of_stream
                for s in off:
                    eng.set_active(False, int(s), 1)
                for s in on:
                    eng.set_active(True, int(s), 1)
                churn["block_after_wall_ms"], churn["block_after_device_ms"] = timed_block(eng, x, y, stream)[::-1]
                churn["streams_moved"] = int((eng.lane_of_stream != lanes_before).sum())
                churn["second_block_wall_ms"], churn["second_block_device_ms"] = timed_block(eng, x, y, stream)[::-1]
                out["churn_64_pause_64_resume"] = churn
        # the same active streams, with their presets, as an engine of their own
        only = [presets[s] for s in np.flatnonzero(active)]
        xs, ys = x[:n_active], y[:n_active]
        with ox.Engine(n_active, F.stereo, 48000, 4) as eng:
            configure(eng, only, props)
            eng.set_placement("auto")
            out["active_only_engine_ms"], _, out["active_only_engine_kernel"] = steady(eng, xs, ys, stream)
        out["ratio"] = out["auto_ms"] / out["active_only_engine_ms"]
        runs.append(out)
    return runs


def caller_run(x, y, stream):
    """One preset (the chain's defaults), whole tiles paused."""
    out = {}
    with ox.Engine(STREAMS, F.stereo, 48000, 4) as eng:
        for i, t in enumerate(CHAIN + [T.eax_reverb]):
            eng.set_effect(i, t)
        for t in range(STREAMS // 32):
            if t % 4 != 0:
                eng.set_active(False, t * 32, 32)
        out["three_quarters_paused_ms"], out["three_quarters_paused_launches_per_block"], out["three_quarters_paused_kernel"] = \
            steady(eng, x, y, stream)
    n = STREAMS // 4
    with ox.Engine(n, F.stereo, 48000, 4) as eng:
        for i, t in enumerate(CHAIN + [T.eax_reverb]):
            eng.set_effect(i, t)
        out["engine_16384_ms"], _, out["engine_16384_kernel"] = steady(eng, x[:n], y[:n], stream)
    out["ratio"] = out["three_quarters_paused_ms"] / out["engine_16384_ms"]
    return out


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(STREAMS)
    x = torch.rand(STREAMS, BLOCK, 2, device=dev, generator=gen) - 0.5
    y = torch.empty_like(x)
    stream = torch.cuda.current_stream().cuda_stream
    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "", "block_frames": BLOCK,
              "chain": "equalizer+chorus+echo+eax_reverb", "auto_113_presets_s_mod_113": auto_runs(x, y, stream),
              "caller_one_preset": caller_run(x, y, stream)}
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()

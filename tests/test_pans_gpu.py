"""Bus formats and pan routes on the GPU: the pan kernels of k_bus.cu give bit for bit the numpy model (pan_model.py) on
the downloaded block -- a mono echo engine at 65 536 streams into stereo buses and the cfg4 chain at 16 384 streams into 5.1
buses, two pan routes per stream (64 category buses + 4096 random send buses), a quarter of the streams paused, a ramp over
2.5 blocks -- for both layouts and both placements, repeatably; at the engine's own format scalar routes keep their bits."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from pan_model import Pans
from route_model import Routes
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED
CHAIN = [T.equalizer, T.chorus, T.echo, T.eax_reverb]
KINDS = {"echo_64k_mono_to_stereo": (65536, 256, F.mono, F.stereo), "cfg4_16k_stereo_to_5.1": (16384, 512, F.stereo, F.five_point_one)}
N_BUSES = 64 + 4096


def _engine(lib, kind, placement):
    S, _, fmt, bus_fmt = KINDS[kind]
    if kind.startswith("cfg4"):
        eng = ox.Engine(S, fmt, 48000, 4, lib=lib)
        eng.set_placement(placement)
        for i, t in enumerate(CHAIN):
            eng.set_effect(i, t)
    else:
        eng = ox.Engine(S, fmt, 48000, 1, lib=lib)
        eng.set_placement(placement)
        for p in range(4):
            eng.set_effect(0, T.echo, ox.default_props(T.echo, lib=lib, delay_=0.02 + 0.01 * p), first_stream=p * S // 4, n_streams=S // 4)
    eng.set_bus_format(bus_fmt)
    return eng


def _paused(S, seed):
    rng = np.random.default_rng(seed)
    active = np.ones(S, dtype=bool)
    active[rng.choice(S, S // 4, replace=False)] = False
    return active


def _set_paused(eng, active):
    for s in np.flatnonzero(~active):
        eng.set_active(False, int(s), 1)


def _routes(S, Cb, C, seed):
    """Per stream its category bus (one of 64, by tile) and a random send bus (64 + one of 4096), random pan matrices."""
    rng = np.random.default_rng(seed)
    bus = np.stack([(np.arange(S) // 32) % 64, 64 + rng.integers(0, 4096, S)], axis=1).astype(np.int32)
    pan = (rng.standard_normal((S, 2, Cb, C)) * 0.7).astype(np.float32)
    pan[rng.random(pan.shape) < 0.1] = 0.0
    return bus, pan


def _to_tiled(x):
    S, n, C = x.shape
    return x.reshape(S // 32, 32, n, C).permute(0, 2, 3, 1).contiguous()


def _exact(expect, got, what=""):
    e = np.ascontiguousarray(expect, dtype=np.float32).view(np.uint32)
    g = np.ascontiguousarray(got, dtype=np.float32).view(np.uint32)
    assert e.shape == g.shape, (what, e.shape, g.shape)
    bad = np.flatnonzero(e != g)
    assert bad.size == 0, (what, "mismatches", bad.size, "first", np.unravel_index(bad[0], e.shape), H.max_abs_diff(expect, got))


def _reduce(eng, y, layout, n_buses, frames):
    stream = torch.cuda.current_stream().cuda_stream
    buses = torch.full((n_buses, frames, eng.bus_channels), 3.0, device=y.device)
    eng.reduce_buses(frames, y, buses, layout=layout, stream=stream)
    torch.cuda.synchronize()
    return buses


@pytest.mark.parametrize("kind", list(KINDS))
def test_pan_buses_are_the_model_over_a_ramp(kind):
    """Blocks before, inside, at the end of and after a 2.5-block pan ramp from scalar routes: mix_buses gives the model's
    buses on its own dst, reduce_buses gives them again in both layouts, and CALLER and AUTO placement give the same blocks
    and buses; a second run of the same calls gives the same bits."""
    lib = H.cuda_lib()
    S, frames, _, _ = KINDS[kind]
    dev = torch.device("cuda:0")
    active = _paused(S, 7)
    stream = torch.cuda.current_stream().cuda_stream
    first = {}
    for run, placement in enumerate(("caller", "auto", "caller")):
        gen = torch.Generator(device=dev).manual_seed(S)
        with _engine(lib, kind, placement) as eng:
            C, Cb = eng.channels, eng.bus_channels
            bus, pan = _routes(S, Cb, C, 8)
            xs = [torch.rand(S, frames, C, device=dev, generator=gen) - 0.5 for _ in range(5)]
            model = Pans(S, C, Cb)
            _set_paused(eng, active)
            eng.set_routes(bus[:, :1], np.full((S, 1), 0.5, np.float32))
            model.set_routes(bus[:, :1], np.full((S, 1), 0.5, np.float32))
            y = torch.full_like(xs[0], 1.5)
            eng.mix(xs[0], y, frames=frames, stream=stream)        # the first block consumes the updates
            model.mixed(frames)
            eng.set_route_pans(pan, bus, ramp_frames=frames * 5 // 2)
            model.set_route_pans(pan, bus, ramp_frames=frames * 5 // 2)
            for blk in range(1, 5):
                buses = torch.full((N_BUSES, frames, Cb), 3.0, device=dev)
                eng.mix_buses(xs[blk], y, frames, buses, stream=stream)
                model.mixed(frames)
                torch.cuda.synchronize()
                y_host, b_host = y.cpu().numpy(), buses.cpu().numpy()
                assert not y_host[~active].view(np.uint32).any()
                what = f"{placement} run {run} block {blk}"
                _exact(b_host, _reduce(eng, y, SM, N_BUSES, frames).cpu().numpy(), what + ": reduce again")
                _exact(b_host, _reduce(eng, _to_tiled(y), TILED, N_BUSES, frames).cpu().numpy(), what + ": TILED")
                if blk not in first:
                    first[blk] = (y_host, b_host)
                    _exact(model.buses(y_host, active, N_BUSES), b_host, what + ": model")
                else:
                    _exact(first[blk][0], y_host, what + ": same block")
                    _exact(first[blk][1], b_host, what + ": same buses")


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_scalar_routes_keep_their_bits_at_the_default_format(layout):
    """At the engine's format (set again explicitly) scalar routes give route_model's buses -- the plain routing's bits --
    steady and ramping; into stereo buses a mono engine's scalar routes fill the left channel with the same bits."""
    lib = H.cuda_lib()
    S, frames = 65536, 256
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(9)
    bus = np.stack([(np.arange(S) // 32) % 64, 64 + rng.integers(0, 4096, S)], axis=1).astype(np.int32)
    gain = (rng.standard_normal(bus.shape) * 0.7).astype(np.float32)
    gen = torch.Generator(device=dev).manual_seed(5)
    for fmt in (F.stereo, F.mono):
        C = ox.channel_count(fmt)
        y = torch.rand(S, frames, C, device=dev, generator=gen) - 0.5
        yl = _to_tiled(y) if layout == TILED else y
        with ox.Engine(S, fmt, 48000, 1, lib=lib) as a, ox.Engine(S, fmt, 48000, 1, lib=lib) as b:
            a.set_bus_format(fmt)
            b.set_bus_format(F.stereo)
            model = Routes(S)
            for ramp in (0, frames * 3):
                for e in (a, b):
                    e.set_routes(bus, gain, ramp_frames=ramp)
                model.set_routes(bus, gain, ramp_frames=ramp)
                expect = model.buses(y.cpu().numpy(), np.ones(S, bool), N_BUSES)
                _exact(expect, _reduce(a, yl, layout, N_BUSES, frames).cpu().numpy(), (fmt, ramp))
                got = _reduce(b, yl, layout, N_BUSES, frames).cpu().numpy()
                _exact(expect[:, :, :1], got[:, :, :1], (fmt, ramp, "into stereo"))
                if fmt == F.mono:
                    assert not got[:, :, 1].view(np.uint32).any()


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_odd_long_and_unaligned_calls_are_the_model(layout):
    """The kernels' edges: 5000 frames (three chunks), 37 and 3 frames, a block and bus buffer one float off their 16-byte
    alignment, over a ramp, for mono, stereo and 5.1 engines into buses of another channel count."""
    lib = H.cuda_lib()
    S, n_buses = 2048, 80
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(13)
    for fmt, bus_fmt in ((F.mono, F.stereo), (F.stereo, F.mono), (F.stereo, F.five_point_one), (F.five_point_one, F.seven_point_one)):
        C, Cb = ox.channel_count(fmt), ox.channel_count(bus_fmt)
        with ox.Engine(S, fmt, 48000, 1, lib=lib) as eng:
            eng.set_bus_format(bus_fmt)
            bus = np.stack([rng.choice(n_buses, 2, replace=False) for _ in range(S)]).astype(np.int32)
            pan = (rng.standard_normal((S, 2, Cb, C)) * 0.7).astype(np.float32)
            model = Pans(S, C, Cb)
            eng.mix(np.zeros((S, 16, C), np.float32))
            model.mixed(16)
            eng.set_route_pans(pan, bus, ramp_frames=2600)
            model.set_route_pans(pan, bus, ramp_frames=2600)
            for frames, offset in ((5000, 0), (37, 1), (3, 0), (64, 1)):
                x = torch.rand(S, frames, C, device=dev, generator=torch.Generator(device=dev).manual_seed(frames)) - 0.5
                xl = (_to_tiled(x) if layout == TILED else x).reshape(-1)
                src = torch.cat([torch.zeros(offset, device=dev), xl])[offset:]   # a view `offset` floats into its storage
                store = torch.full((offset + n_buses * frames * Cb,), 3.0, device=dev)
                buses = store[offset:]
                eng.reduce_buses(frames, src, buses, layout=layout, stream=torch.cuda.current_stream().cuda_stream, n_buses=n_buses)
                torch.cuda.synchronize()
                expect = model.buses(x.cpu().numpy(), np.ones(S, bool), n_buses)
                _exact(expect, buses.cpu().numpy().reshape(n_buses, frames, Cb), (fmt, bus_fmt, frames, offset))

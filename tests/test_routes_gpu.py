"""Routes with gains and ramps on the GPU: the weighted level-0 kernels of k_bus.cu give bit for bit the numpy model
(route_model.py) on the downloaded block -- two routes per stream (64 category buses + 4096 random send buses), random
gains, a quarter of the streams paused, a ramp over 2.5 blocks -- for both layouts and both placements, on the cfg4 chain at
16 384 streams and an echo-only engine at 65 536 streams."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from route_model import Routes
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED
CHAIN = [T.equalizer, T.chorus, T.echo, T.eax_reverb]
KINDS = {"cfg4_16k": (16384, 512), "echo_64k": (65536, 256)}   # streams, frames per block
N_BUSES = 64 + 4096


def _engine(lib, kind, placement):
    S, _ = KINDS[kind]
    if kind == "cfg4_16k":
        eng = ox.Engine(S, F.stereo, 48000, 4, lib=lib)
        eng.set_placement(placement)
        for i, t in enumerate(CHAIN):
            eng.set_effect(i, t)
        return eng
    eng = ox.Engine(S, F.stereo, 48000, 1, lib=lib)
    eng.set_placement(placement)
    for p in range(4):
        eng.set_effect(0, T.echo, ox.default_props(T.echo, lib=lib, delay_=0.02 + 0.01 * p), first_stream=p * S // 4, n_streams=S // 4)
    return eng


def _paused(S, seed):
    rng = np.random.default_rng(seed)
    active = np.ones(S, dtype=bool)
    active[rng.choice(S, S // 4, replace=False)] = False
    return active


def _set_paused(eng, active):
    for s in np.flatnonzero(~active):
        eng.set_active(False, int(s), 1)


def _routes(S, seed):
    """Per stream its category bus (one of 64, by tile) and a random send bus (64 + one of 4096), random gains."""
    rng = np.random.default_rng(seed)
    bus = np.stack([(np.arange(S) // 32) % 64, 64 + rng.integers(0, 4096, S)], axis=1).astype(np.int32)
    gain = (rng.standard_normal(bus.shape) * 0.7).astype(np.float32)
    gain[rng.random(bus.shape) < 0.05] = 0.0
    return bus, gain


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
    buses = torch.full((n_buses, frames, 2), 3.0, device=y.device)
    eng.reduce_buses(frames, y, buses, layout=layout, stream=stream)
    torch.cuda.synchronize()
    return buses


@pytest.mark.parametrize("kind", list(KINDS))
def test_weighted_buses_are_the_model_over_a_ramp(kind):
    """Blocks before, inside, at the end of and after a 2.5-block ramp: mix_buses gives the model's buses on its own dst,
    reduce_buses gives them again in both layouts, and CALLER and AUTO placement give the same blocks and buses."""
    lib = H.cuda_lib()
    S, frames = KINDS[kind]
    dev = torch.device("cuda:0")
    active = _paused(S, 7)
    bus, gain = _routes(S, 8)
    stream = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device=dev).manual_seed(S)
    xs = [torch.rand(S, frames, 2, device=dev, generator=gen) - 0.5 for _ in range(5)]
    first = {}
    for placement in ("caller", "auto"):
        model = Routes(S)
        with _engine(lib, kind, placement) as eng:
            _set_paused(eng, active)
            y = torch.full_like(xs[0], 1.5)
            eng.mix(xs[0], y, frames=frames, stream=stream)        # the first block consumes the updates
            model.mixed(frames)
            eng.set_routes(bus, gain, ramp_frames=frames * 5 // 2)
            model.set_routes(bus, gain, ramp_frames=frames * 5 // 2)
            for blk in range(1, 5):
                buses = torch.full((N_BUSES, frames, 2), 3.0, device=dev)
                eng.mix_buses(xs[blk], y, frames, buses, stream=stream)
                model.mixed(frames)
                torch.cuda.synchronize()
                y_host, b_host = y.cpu().numpy(), buses.cpu().numpy()
                assert not y_host[~active].view(np.uint32).any()
                what = f"{placement} block {blk}"
                _exact(b_host, _reduce(eng, y, SM, N_BUSES, frames).cpu().numpy(), what + ": reduce again")
                _exact(b_host, _reduce(eng, _to_tiled(y), TILED, N_BUSES, frames).cpu().numpy(), what + ": TILED")
                if blk not in first:
                    first[blk] = (y_host, b_host)
                    _exact(model.buses(y_host, active, N_BUSES), b_host, what + ": model")
                else:
                    _exact(first[blk][0], y_host, what + ": CALLER vs AUTO block")
                    _exact(first[blk][1], b_host, what + ": CALLER vs AUTO buses")


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_a_unity_plan_is_route_streams(layout):
    lib = H.cuda_lib()
    S, frames = KINDS["echo_64k"]
    dev = torch.device("cuda:0")
    bus, _ = _routes(S, 9)
    routing = bus[:, 1].copy()
    routing[::9] = ox.BUS_NONE
    gen = torch.Generator(device=dev).manual_seed(5)
    y = torch.rand(S, frames, 2, device=dev, generator=gen) - 0.5
    if layout == TILED:
        y = _to_tiled(y)
    with ox.Engine(S, F.stereo, 48000, 1, lib=lib) as a, ox.Engine(S, F.stereo, 48000, 1, lib=lib) as b:
        a.route(routing)
        b.set_routes(routing[:, None], np.ones((S, 1), np.float32))
        _exact(_reduce(a, y, layout, N_BUSES, frames).cpu().numpy(), _reduce(b, y, layout, N_BUSES, frames).cpu().numpy())


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_weighted_mix_buses_leaves_the_block_and_kernel_of_mix(kind, layout):
    lib = H.cuda_lib()
    S, frames = KINDS[kind]
    dev = torch.device("cuda:0")
    active = _paused(S, 9)
    bus, gain = _routes(S, 10)
    stream = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device=dev).manual_seed(3)
    with _engine(lib, kind, "caller") as a, _engine(lib, kind, "caller") as b:
        for eng in (a, b):
            _set_paused(eng, active)
            eng.set_routes(bus, gain, ramp_frames=frames * 3 // 2)
        for blk in range(2):
            x = torch.rand(S, frames, 2, device=dev, generator=gen) - 0.5
            if layout == TILED:
                x = _to_tiled(x)
            ya, yb = torch.full_like(x, 1.5), torch.full_like(x, 1.5)
            buses = torch.full((N_BUSES, frames, 2), 3.0, device=dev)
            a.mix_buses(x, ya, frames, buses, layout=layout, stream=stream)
            b.mix(x, yb, frames=frames, layout=layout, stream=stream)
            torch.cuda.synchronize()
            assert torch.equal(ya.view(torch.int32), yb.view(torch.int32)), blk
            assert a.last_kernel == b.last_kernel, (a.last_kernel, b.last_kernel)
            again = _reduce(b, yb, layout, N_BUSES, frames)
            assert torch.equal(buses.view(torch.int32), again.view(torch.int32)), blk

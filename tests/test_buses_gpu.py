"""Submix buses on the GPU: the sm_100a kernels of k_bus.cu give bit for bit the numpy model of the summation order
(bus_model.py) on the downloaded block, for both layouts, both placements and a quarter of the streams paused, on the
cfg4 chain at 16 384 streams and an echo-only engine at 65 536 streams."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from bus_model import model_buses
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED
CHAIN = [T.equalizer, T.chorus, T.echo, T.eax_reverb]
KINDS = {"cfg4_16k": (16384, 512), "echo_64k": (65536, 256)}   # streams, frames per block


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
    for p in range(4):   # four echo presets on whole tiles: placement keeps them, AUTO packs the paused streams apart
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


def _routings(S, seed):
    rng = np.random.default_rng(seed)
    rand = rng.integers(0, 4096, S).astype(np.int32)
    rand[rng.random(S) < 0.1] = ox.BUS_NONE
    skew = np.empty(S, dtype=np.int32)
    half = rng.permutation(S)
    skew[half[: S // 2]] = 0
    skew[half[S // 2:]] = 1 + np.arange(S - S // 2)
    return {
        "one_bus": (np.zeros(S, np.int32), 1),
        "64_tile_buses": (((np.arange(S) // 32) % 64).astype(np.int32), 64),
        "4096_random": (rand, 4096),
        "bus_per_stream": (np.arange(S, dtype=np.int32), S),
        "skew": (skew, 1 + S - S // 2),
    }


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
def test_buses_are_the_model_for_every_routing_layout_and_placement(kind):
    """Per routing: the buses of the same mixed block are bit-exact against the model, identical from call to call,
    identical for STREAM_MAJOR and TILED, and identical for CALLER and AUTO placement (whose blocks are identical)."""
    lib = H.cuda_lib()
    S, frames = KINDS[kind]
    dev = torch.device("cuda:0")
    active = _paused(S, 7)
    routings = _routings(S, 8)
    gen = torch.Generator(device=dev).manual_seed(S)
    x = torch.rand(S, frames, 2, device=dev, generator=gen) - 0.5
    stream = torch.cuda.current_stream().cuda_stream
    first = {}
    y_ref = None
    for placement in ("caller", "auto"):
        with _engine(lib, kind, placement) as eng:
            _set_paused(eng, active)
            y = torch.full_like(x, 1.5)
            for _ in range(2):   # the second block runs past the updates of the first
                eng.mix(x, y, frames=frames, stream=stream)
            torch.cuda.synchronize()
            y_host = y.cpu().numpy()
            assert not y_host[~active].view(np.uint32).any()
            if y_ref is None:
                y_ref = y_host
            _exact(y_ref, y_host, f"{placement}: block")
            yt = _to_tiled(y)
            for name, (routing, n_buses) in routings.items():
                eng.route(routing)
                b_sm = _reduce(eng, y, SM, n_buses, frames).cpu().numpy()
                _exact(b_sm, _reduce(eng, y, SM, n_buses, frames).cpu().numpy(), f"{placement} {name}: run to run")
                _exact(b_sm, _reduce(eng, yt, TILED, n_buses, frames).cpu().numpy(), f"{placement} {name}: TILED")
                if name not in first:
                    first[name] = b_sm
                    _exact(model_buses(y_host, routing, active, n_buses), b_sm, f"{placement} {name}: model")
                else:
                    _exact(first[name], b_sm, f"{placement} {name}: CALLER vs AUTO")
    assert set(first) == set(routings)


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_mix_buses_leaves_the_block_and_kernel_of_mix(kind, layout):
    """mix_buses over two blocks (4096 random buses, a quarter paused): dst and last_kernel as from mix on a twin engine,
    buses as reduce_buses of that dst."""
    lib = H.cuda_lib()
    S, frames = KINDS[kind]
    dev = torch.device("cuda:0")
    active = _paused(S, 9)
    routing, n_buses = _routings(S, 10)["4096_random"]
    stream = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device=dev).manual_seed(3)
    with _engine(lib, kind, "caller") as a, _engine(lib, kind, "caller") as b:
        for eng in (a, b):
            _set_paused(eng, active)
            eng.route(routing)
        for blk in range(2):
            x = torch.rand(S, frames, 2, device=dev, generator=gen) - 0.5
            if layout == TILED:
                x = _to_tiled(x)
            ya, yb = torch.full_like(x, 1.5), torch.full_like(x, 1.5)
            buses = torch.full((n_buses, frames, 2), 3.0, device=dev)
            a.mix_buses(x, ya, frames, buses, layout=layout, stream=stream)
            b.mix(x, yb, frames=frames, layout=layout, stream=stream)
            torch.cuda.synchronize()
            assert torch.equal(ya.view(torch.int32), yb.view(torch.int32)), blk
            assert a.last_kernel == b.last_kernel, (a.last_kernel, b.last_kernel)
            again = _reduce(b, yb, layout, n_buses, frames)
            assert torch.equal(buses.view(torch.int32), again.view(torch.int32)), blk

"""Submix buses (oalsfx_engine_route_streams / reduce_buses / mix_buses) on the CPU build of the engine (tests/_build):
bit-exact against the numpy model of the summation order (bus_model.py) and independent of layout, placement, activity
history and the cut of a call into blocks."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from bus_model import model_buses
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED


def _rows(S, frames, C, seed):
    """[S][frames][C] float32 of mixed magnitudes and signs, with some -0.0f and exact cancellations."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((S, frames, C)) * 10.0 ** rng.integers(-3, 4, (S, 1, 1))).astype(np.float32)
    x[rng.random(x.shape) < 0.02] = np.float32(-0.0)
    x[1::7] = -x[0:-1:7][: len(x[1::7])]
    return x


def _to_layout(x, layout):
    if layout == SM:
        return np.ascontiguousarray(x)
    S, frames, C = x.shape
    T_ = (S + 31) // 32
    t = np.full((T_ * 32, frames, C), np.float32(7.0))   # padding lanes hold garbage: they are never members
    t[:S] = x
    return np.ascontiguousarray(t.reshape(T_, 32, frames, C).transpose(0, 2, 3, 1))


def _from_layout(y, S, layout):
    if layout == SM:
        return y
    T_, frames, C, _ = y.shape
    return y.transpose(0, 3, 1, 2).reshape(T_ * 32, frames, C)[:S]


def _reduce(eng, x, layout, n_buses):
    frames, C = x.shape[1], x.shape[2]
    buses = np.full((n_buses, frames, C), np.float32(3.0))
    eng.reduce_buses(frames, _to_layout(x, layout), buses, layout=layout)
    return buses


def _exact(expect, got, what=""):
    assert expect.shape == got.shape, (what, expect.shape, got.shape)
    bad = np.flatnonzero(expect.view(np.uint32) != got.view(np.uint32))
    assert bad.size == 0, (what, "mismatches", bad.size, "first", np.unravel_index(bad[0], expect.shape), H.max_abs_diff(expect, got))


def _random_routing(rng, S, n_buses, unrouted=0.1):
    r = rng.integers(0, n_buses, S).astype(np.int32)
    r[rng.random(S) < unrouted] = ox.BUS_NONE
    return r


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("fmt", [F.mono, F.stereo, F.five_point_one], ids=["mono", "stereo", "5.1"])
def test_buses_match_the_model(fmt, layout):
    """150 streams (ragged last tile): random routing over 12 buses with unrouted streams and empty buses, every stream
    on its own bus, and more buses than needed; odd frame counts."""
    lib = H.emu_lib()
    S = 150
    rng = np.random.default_rng(int(fmt) * 10 + layout)
    active = np.ones(S, dtype=bool)
    with ox.Engine(S, fmt, 48000, 1, lib=lib) as eng:
        C = eng.channels
        routing = _random_routing(rng, S, 12)
        routing[routing == 5] = 6                       # bus 5 is empty
        routings = [(routing, 12), (np.arange(S, dtype=np.int32), S), (routing, 40)]
        for i, (r, n_buses) in enumerate(routings):
            eng.route(r)
            for frames in (37, 1, 64):
                x = _rows(S, frames, C, 100 * i + frames)
                _exact(model_buses(x, r, active, n_buses), _reduce(eng, x, layout, n_buses), (i, frames))
        assert not _reduce(eng, _rows(S, 9, C, 1), layout, 40)[12:].view(np.uint32).any()   # buses nobody is routed to: +0.0f


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_a_bus_of_more_than_1024_members_takes_three_levels(layout):
    lib = H.emu_lib()
    S = 1100
    routing = np.zeros(S, dtype=np.int32)
    routing[::50] = 1
    routing[3] = ox.BUS_NONE
    with ox.Engine(S, F.stereo, 48000, 1, lib=lib) as eng:
        eng.route(routing)
        assert (routing == 0).sum() > 1024
        x = _rows(S, 5, 2, 3)
        _exact(model_buses(x, routing, np.ones(S, bool), 2), _reduce(eng, x, layout, 2))


def test_a_long_call_equals_one_call_per_block_and_layouts_agree():
    """5000 frames in one call (chunks of 2048 inside) equal three calls of 2048 / 2048 / 904 frames, and the model."""
    lib = H.emu_lib()
    S = 70
    rng = np.random.default_rng(5)
    routing = _random_routing(rng, S, 6)
    with ox.Engine(S, F.stereo, 48000, 1, lib=lib) as eng:
        eng.route(routing)
        x = _rows(S, 5000, 2, 8)
        whole = _reduce(eng, x, SM, 6)
        _exact(whole, _reduce(eng, x, TILED, 6), "tiled")
        parts = [_reduce(eng, np.ascontiguousarray(x[:, a:b]), SM, 6) for a, b in ((0, 2048), (2048, 4096), (4096, 5000))]
        _exact(np.concatenate(parts, axis=1), whole, "blocks")
        _exact(model_buses(x, routing, np.ones(S, bool), 6), whole, "model")


def _echo_engine(lib, S, placement, presets=7):
    eng = ox.Engine(S, F.stereo, 48000, 1, lib=lib)
    eng.set_placement(placement)
    for s in range(S):
        eng.set_effect(0, T.echo, ox.default_props(T.echo, lib=lib, delay_=0.01 + 0.002 * (s % presets)), first_stream=s, n_streams=1)
    return eng


def _noise(S, frames, seed):
    return np.stack([H.noise(seed + s, 2, frames) for s in range(S)])


def test_paused_streams_are_not_members_and_placements_agree():
    """Streams pause and resume between blocks; the buses of each block are the model over the streams active at that
    call, the same for CALLER and AUTO placement (where pausing moves lanes) and for both layouts."""
    lib = H.emu_lib()
    S = 90
    rng = np.random.default_rng(9)
    routing = _random_routing(rng, S, 5)
    engines = [_echo_engine(lib, S, p) for p in ("caller", "auto")]
    try:
        for eng in engines:
            eng.route(routing)
        active = np.ones(S, dtype=bool)
        for b in range(4):
            if b > 0:
                flip = rng.choice(S, 20, replace=False)
                active[flip] = ~active[flip]
                for eng in engines:
                    for s in flip:
                        eng.set_active(bool(active[s]), int(s), 1)
            x = _noise(S, 48, 10 * b)
            results = []
            for eng in engines:
                y = eng.mix(x)
                assert not y[~active].view(np.uint32).any()
                for layout in (SM, TILED):
                    results.append(_reduce(eng, y, layout, 5))
                _exact(model_buses(y, routing, active, 5), results[-1], b)
            for r in results[1:]:
                _exact(results[0], r, b)
        # pausing / resuming alone changes the buses of the next call on the same block
        routed = np.flatnonzero(routing >= 0)
        s0, s1 = int(routed[np.flatnonzero(active[routed])[0]]), int(routed[np.flatnonzero(~active[routed])[0]])
        before = _reduce(engines[1], y, SM, 5)
        for eng in engines:
            eng.set_active(False, s0, 1)
            eng.set_active(True, s1, 1)
        active[s0], active[s1] = False, True
        after = [_reduce(eng, y, TILED, 5) for eng in engines]
        assert not np.array_equal(before, after[0])
        for got in after:
            _exact(model_buses(y, routing, active, 5), got, "after a toggle")
        # the rows of paused streams are never read
        x = _rows(S, 16, 2, 4)
        junk = x.copy()
        junk[~active] = np.float32(1e30)
        _exact(_reduce(engines[0], x, SM, 5), _reduce(engines[0], junk, SM, 5), "paused rows read")
    finally:
        for eng in engines:
            eng.close()


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_mix_buses_is_mix_then_reduce_buses(layout):
    lib = H.emu_lib()
    S = 75
    routing = _random_routing(np.random.default_rng(2), S, 4)
    a, b = _echo_engine(lib, S, "caller"), _echo_engine(lib, S, "caller")
    try:
        a.route(routing)
        b.route(routing)
        for blk, frames in enumerate((64, 33)):
            x = _to_layout(_noise(S, frames, 7 * blk), layout)
            ya, yb = np.full_like(x, 1.5), np.full_like(x, 1.5)
            buses = np.full((4, frames, 2), np.float32(3.0))
            a.mix_buses(x, ya, frames, buses, layout=layout)
            b.mix(x, yb, frames=frames, layout=layout, space=ox.SPACE_DEVICE)
            _exact(yb, ya, "dst")
            _exact(_reduce(b, _from_layout(yb, S, layout), layout, 4), buses, "buses")
            assert a.last_kernel == b.last_kernel
    finally:
        a.close()
        b.close()


def test_routing_survives_reset_placement_and_restore():
    lib = H.emu_lib()
    S = 64
    routing = _random_routing(np.random.default_rng(4), S, 3)
    with _echo_engine(lib, S, "caller") as eng, _echo_engine(lib, S, "caller") as fresh:
        size = eng.snapshot().size
        eng.route(routing)
        assert eng.snapshot().size == size
        y = eng.mix(_noise(S, 32, 0))
        expect = model_buses(y, routing, np.ones(S, bool), 3)
        snap = eng.snapshot()
        eng.reset(0, S)
        _exact(expect, _reduce(eng, y, SM, 3), "after reset_streams")
        eng.set_placement("auto")
        _exact(expect, _reduce(eng, y, TILED, 3), "after AUTO")
        eng.set_placement("caller")
        _exact(expect, _reduce(eng, y, SM, 3), "after CALLER")
        eng.restore(fresh.snapshot())      # a snapshot of an engine routed to bus 0 only
        _exact(expect, _reduce(eng, y, SM, 3), "after restore")
        fresh.restore(snap)
        _exact(model_buses(y, np.zeros(S, np.int32), np.ones(S, bool), 1), _reduce(fresh, y, SM, 1), "restore keeps the routing")


def test_bad_arguments_are_argument_errors_and_a_refused_mix_buses_mixes_nothing():
    lib = H.emu_lib()
    S = 40
    with _echo_engine(lib, S, "caller") as eng, _echo_engine(lib, S, "caller") as twin:
        routing = np.full(S, 2, dtype=np.int32)
        routing[0] = ox.BUS_NONE
        for first, bus in ((-1, [0]), (40, [0]), (39, [0, 0]), (0, [-2])):
            with pytest.raises(ox.OalsfxError) as err:
                eng.route(np.array(bus), first_stream=first)
            assert err.value.code == -1
        with pytest.raises(ox.OalsfxError):
            eng.route(np.array([], dtype=np.int32))
        assert lib.oalsfx_engine_route_streams(eng._h, 0, 1, None) == -1
        eng.route(routing)
        twin.route(routing)
        x = _noise(S, 16, 1)
        y = np.empty_like(x)
        buses = np.zeros((3, 16, 2), np.float32)
        bad = [
            dict(frames=0), dict(frames=-4), dict(layout=7), dict(n_buses=0), dict(n_buses=2), dict(src=None),
            dict(dst=None), dict(buses=None),
        ]
        for b in bad:
            a = dict(frames=16, src=x.ctypes.data, dst=y.ctypes.data, layout=SM, n_buses=3, buses=buses.ctypes.data)
            a.update(b)
            rc = lib.oalsfx_engine_mix_buses(eng._h, a["frames"], a["src"], a["dst"], a["layout"], a["n_buses"], a["buses"], None)
            assert rc == -1, b
            if "src" not in b:
                rc = lib.oalsfx_engine_reduce_buses(eng._h, a["frames"], a["dst"], a["layout"], a["n_buses"], a["buses"], None)
                assert rc == -1, b
        # the refused calls advanced nothing: the next block equals that of an engine that never saw them
        x2 = _noise(S, 16, 2)
        _exact(twin.mix(x2), eng.mix(x2), "state advanced by a refused call")


def test_two_half_engines_sum_to_the_whole():
    """Each rank holds half of the streams; the sum of their buses (the all-reduce) is the one-engine buses up to
    reassociation."""
    lib = H.emu_lib()
    S, half = 256, 128
    routing = _random_routing(np.random.default_rng(6), S, 8)
    x = _noise(S, 24, 11)
    with ox.Engine(S, F.stereo, 48000, 1, lib=lib) as whole, ox.Engine(half, F.stereo, 48000, 1, lib=lib) as a, \
            ox.Engine(half, F.stereo, 48000, 1, lib=lib) as b:
        whole.route(routing)
        a.route(routing[:half])
        b.route(routing[half:])
        one = _reduce(whole, x, SM, 8)
        two = _reduce(a, x[:half], SM, 8) + _reduce(b, x[half:], SM, 8)
        assert np.abs(one.astype(np.float64) - two).max() <= 1e-5 * np.sqrt(S)

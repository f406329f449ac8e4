"""Routes with gains and ramps (oalsfx_engine_set_routes) on the CPU build of the engine (tests/_build): bit-exact against
the numpy model (route_model.py) on the uint32 images, independent of layout, placement and the cut of a call into blocks,
and following the frame clock through mixes, pauses, resets, placement switches and restores."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from bus_model import model_buses
from route_model import Routes, gain_at
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED
F32 = np.float32


def _rows(S, frames, C, seed):
    """[S][frames][C] float32 of mixed magnitudes and signs, with some -0.0f and exact cancellations."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((S, frames, C)) * 10.0 ** rng.integers(-3, 4, (S, 1, 1))).astype(F32)
    x[rng.random(x.shape) < 0.02] = F32(-0.0)
    x[1::7] = -x[0:-1:7][: len(x[1::7])]
    return x


def _to_layout(x, layout):
    if layout == SM:
        return np.ascontiguousarray(x)
    S, frames, C = x.shape
    t = np.full(((S + 31) // 32 * 32, frames, C), F32(7.0))   # padding lanes hold garbage: they are never members
    t[:S] = x
    return np.ascontiguousarray(t.reshape(-1, 32, frames, C).transpose(0, 2, 3, 1))


def _reduce(eng, x, layout, n_buses):
    frames, C = x.shape[1], x.shape[2]
    buses = np.full((n_buses, frames, C), F32(3.0))
    eng.reduce_buses(frames, _to_layout(x, layout), buses, layout=layout)
    return buses


def _exact(expect, got, what=""):
    assert expect.shape == got.shape, (what, expect.shape, got.shape)
    bad = np.flatnonzero(expect.view(np.uint32) != got.view(np.uint32))
    assert bad.size == 0, (what, "mismatches", bad.size, "first", np.unravel_index(bad[0], expect.shape), H.max_abs_diff(expect, got))


def _random_routes(rng, S, R, n_buses, none=0.15):
    """[S][R] distinct buses per stream (some BUS_NONE) and gains: negative, zero, tiny and ordinary."""
    bus = np.stack([rng.choice(n_buses, R, replace=False) for _ in range(S)]).astype(np.int32)
    bus[rng.random(bus.shape) < none] = ox.BUS_NONE
    gain = (rng.standard_normal(bus.shape) * 2).astype(F32)
    gain[rng.random(bus.shape) < 0.1] = F32(0.0)
    gain[rng.random(bus.shape) < 0.05] = F32(1e-30)
    gain[rng.random(bus.shape) < 0.1] = F32(1.0)
    return bus, gain


def _echo_engine(lib, S, placement="caller", presets=7):
    eng = ox.Engine(S, F.stereo, 48000, 1, lib=lib)
    eng.set_placement(placement)
    for s in range(S):
        eng.set_effect(0, T.echo, ox.default_props(T.echo, lib=lib, delay_=0.01 + 0.002 * (s % presets)), first_stream=s, n_streams=1)
    return eng


def _noise(S, frames, seed):
    return np.stack([H.noise(seed + s, 2, frames) for s in range(S)])


def _mix_buses(eng, x, n_buses, layout=SM):
    S, frames, C = x.shape
    xl = _to_layout(x, layout)
    y = np.full_like(xl, 1.5)
    buses = np.full((n_buses, frames, C), F32(3.0))
    eng.mix_buses(xl, y, frames, buses, layout=layout)
    if layout == TILED:
        y = y.transpose(0, 3, 1, 2).reshape(-1, frames, C)[:S]
    return np.ascontiguousarray(y), buses


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("fmt", [F.mono, F.stereo, F.five_point_one], ids=["mono", "stereo", "5.1"])
def test_routes_match_the_model(fmt, layout):
    """150 streams (ragged last tile), 1..4 routes per stream over 12 buses with unrouted streams and an empty bus, gains
    negative / zero / tiny; a zero-gain route of a stream holding an Inf puts NaN on its bus, as the model does."""
    lib = H.emu_lib()
    S = 150
    rng = np.random.default_rng(int(fmt) * 10 + layout)
    active = np.ones(S, dtype=bool)
    with ox.Engine(S, fmt, 48000, 1, lib=lib) as eng:
        C = eng.channels
        model = Routes(S)
        for R in (1, 2, 3, 4):
            bus, gain = _random_routes(rng, S, R, 12)
            bus[bus == 5] = ox.BUS_NONE                      # bus 5 is empty
            eng.set_routes(bus, gain)
            model.set_routes(bus, gain)
            for frames in (37, 1, 64):
                x = _rows(S, frames, C, 100 * R + frames)
                _exact(model.buses(x, active, 12), _reduce(eng, x, layout, 12), (R, frames))
        s = int(np.flatnonzero((bus >= 0).any(axis=1))[0])
        zero = np.where(bus[s] >= 0, F32(0.0), gain[s])
        eng.set_routes(bus[s:s + 1], zero[None], first_stream=s)
        model.set_routes(bus[s:s + 1], zero[None], first_stream=s)
        x = _rows(S, 8, C, 3)
        x[s, 2, 0] = np.inf
        got = _reduce(eng, x, layout, 12)
        _exact(model.buses(x, active, 12), got, "0 * Inf")
        assert np.isnan(got[bus[s][bus[s] >= 0], 2, 0]).all()


def test_unity_routes_are_route_streams_and_route_streams_drops_extra_routes():
    lib = H.emu_lib()
    S = 100
    rng = np.random.default_rng(1)
    routing = rng.integers(-1, 9, S).astype(np.int32)
    with _echo_engine(lib, S) as a, _echo_engine(lib, S) as b:
        a.route(routing)
        b.set_routes(routing[:, None], np.ones((S, 1), F32))
        for blk in range(2):
            x = _noise(S, 40, blk)
            for layout in (SM, TILED):
                ya, ba = _mix_buses(a, x, 9, layout)
                yb, bb = _mix_buses(b, x, 9, layout)
                _exact(ya, yb, "dst")
                _exact(ba, bb, "unity set_routes")
        extra = np.stack([routing, (routing + 1) % 9], axis=1)
        b.set_routes(extra, np.full(extra.shape, 0.5, F32), ramp_frames=50)
        b.route(routing)
        for layout in (SM, TILED):
            x = _noise(S, 40, 9)
            _exact(_mix_buses(a, x, 9, layout)[1], _mix_buses(b, x, 9, layout)[1], "route_streams after multi-routes")


def test_a_change_without_ramp_applies_to_the_block_already_mixed():
    """route_streams and set_routes with ramp_frames = 0 after a mix: reducing that block uses the new routes and gains."""
    lib = H.emu_lib()
    S = 64
    rng = np.random.default_rng(12)
    with _echo_engine(lib, S) as eng:
        y = eng.mix(_noise(S, 32, 3))
        routing = rng.integers(0, 6, S).astype(np.int32)
        eng.route(routing)
        _exact(model_buses(y, routing, np.ones(S, bool), 6), _reduce(eng, y, SM, 6), "route_streams")
        bus, gain = _random_routes(rng, S, 3, 6)
        eng.set_routes(bus, gain)
        model = Routes(S)
        model.mixed(32)
        model.set_routes(bus, gain)
        _exact(model.buses(y, np.ones(S, bool), 6), _reduce(eng, y, TILED, 6), "set_routes")


def test_a_ramp_over_blocks_is_the_model_and_one_long_call():
    """A 300-frame ramp over mix_buses blocks of 128 / 64 / 37 frames; the same frames as one call give the same bits."""
    lib = H.emu_lib()
    S, n_buses = 70, 10
    rng = np.random.default_rng(3)
    bus, gain = _random_routes(rng, S, 2, n_buses)
    blocks = [128, 64, 37, 128, 64]
    x = _noise(S, sum(blocks), 5)
    with _echo_engine(lib, S) as eng, _echo_engine(lib, S) as whole:
        model = Routes(S)
        warm = _noise(S, 16, 99)
        for e in (eng, whole):
            e.mix(warm)
            e.set_routes(bus, gain, ramp_frames=300)
        model.mixed(16)
        model.set_routes(bus, gain, ramp_frames=300)
        got, f0 = [], 0
        for n in blocks:
            layout = TILED if len(got) % 2 else SM
            y, buses = _mix_buses(eng, np.ascontiguousarray(x[:, f0:f0 + n]), n_buses, layout)
            model.mixed(n)
            _exact(model.buses(y, np.ones(S, bool), n_buses), buses, ("block", len(got)))
            got.append(buses)
            f0 += n
        _, one = _mix_buses(whole, x, n_buses)
        _exact(np.concatenate(got, axis=1), one, "one long call")


def test_ramp_starts_follow_the_last_mixed_frame():
    """Rows of ones read the gains off the bus.  A change mid-ramp starts from the gain of the last mixed frame; two changes
    without a mix between restart from the same g0; a new route fades in from 0."""
    lib = H.emu_lib()
    S = 3
    ones = np.ones((S, 10, 1), F32)
    with ox.Engine(S, F.mono, 48000, 1, lib=lib) as eng, ox.Engine(S, F.mono, 48000, 1, lib=lib) as twin:
        def block(e, n):   # mix n frames (the clock moves on), then the buses of a block of ones: the gains
            e.mix(np.zeros((S, n, 1), F32))
            return _reduce(e, np.ascontiguousarray(ones[:, :n]), SM, 3)[:, :, 0]
        for e in (eng, twin):
            e.route(np.array([0, 1, 2], np.int32))
            e.set_routes([[0]], [[F32(0.0)]], first_stream=0)
            block(e, 10)
            e.set_routes([[0]], [[F32(1.0)]], first_stream=0, ramp_frames=4)   # 0 -> 1 over 4 frames
        b = block(eng, 2)
        assert list(b[0]) == [0.25, 0.5]
        eng.set_routes([[0]], [[F32(-1.0)]], first_stream=0, ramp_frames=3)    # mid-ramp: from 0.5
        b = block(eng, 4)
        g = gain_at(F32(0.5), F32(-1.0), 3, 12, 12 + np.arange(4))
        _exact(g, b[0], "mid-ramp change")
        assert b[0][-1] == -1.0
        # two changes with no mix between: the second starts from the first's g0, i.e. where the route stood
        twin.set_routes([[0]], [[F32(1.0)]], first_stream=0, ramp_frames=4)
        twin.set_routes([[0]], [[F32(2.0)]], first_stream=0, ramp_frames=4)
        tb = block(twin, 2)
        _exact(gain_at(F32(0.0), F32(2.0), 4, 10, np.array([10, 11])), tb[0], "restart from the same g0")
        # a new route fades in from 0; the removed stream-2 route stops at once
        eng.set_routes([[1, 2]], [[F32(2.0), F32(1.0)]], first_stream=1, ramp_frames=8)
        eng.set_routes([[ox.BUS_NONE]], first_stream=2)
        b = block(eng, 4)
        _exact(gain_at(F32(0.0), F32(1.0), 8, 16, 16 + np.arange(4)), b[2], "fade-in of a new route")
        assert b[1][0] == F32(1.0) + (F32(2.0) - F32(1.0)) * (F32(1) / F32(8))


def test_reduce_after_mix_is_mix_buses_and_repeats_during_a_ramp():
    lib = H.emu_lib()
    S, n_buses = 66, 6
    bus, gain = _random_routes(np.random.default_rng(8), S, 3, n_buses)
    with _echo_engine(lib, S) as a, _echo_engine(lib, S) as b:
        for e in (a, b):
            e.set_routes(bus, gain, ramp_frames=100)
        for blk, n in enumerate((48, 48, 48)):
            x = _noise(S, n, 20 + blk)
            ya, ba = _mix_buses(a, x, n_buses)
            yb = b.mix(x)
            _exact(ya, yb, "dst")
            _exact(ba, _reduce(b, yb, SM, n_buses), "reduce after mix")
            for layout in (SM, TILED, SM):
                _exact(ba, _reduce(b, yb, layout, n_buses), ("again", layout))


@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_paused_streams_are_not_members_and_their_ramps_run_on(placement):
    """Streams pause and resume during a ramp: the buses are the model over the active streams with the gains of the
    clock, for both placements; paused rows are never read (NaN there would show)."""
    lib = H.emu_lib()
    S, n_buses = 90, 7
    rng = np.random.default_rng(11)
    bus, gain = _random_routes(rng, S, 2, n_buses)
    with _echo_engine(lib, S, placement) as eng, _echo_engine(lib, S, "caller") as ref:
        model = Routes(S)
        active = np.ones(S, dtype=bool)
        for e in (eng, ref):
            e.set_routes(bus, gain, ramp_frames=200)
        model.set_routes(bus, gain, ramp_frames=200)
        for blk in range(5):
            if blk > 0:
                flip = rng.choice(S, 15, replace=False)
                active[flip] = ~active[flip]
                for e in (eng, ref):
                    for s in flip:
                        e.set_active(bool(active[s]), int(s), 1)
            x = _noise(S, 48, 30 + blk)
            y, buses = _mix_buses(eng, x, n_buses, TILED if blk % 2 else SM)
            _, ref_buses = _mix_buses(ref, x, n_buses)
            model.mixed(48)
            _exact(model.buses(y, active, n_buses), buses, blk)
            _exact(ref_buses, buses, ("CALLER vs", placement))
            junk = y.copy()
            junk[~active] = np.nan
            _exact(buses, _reduce(eng, junk, SM, n_buses), "paused rows read")


def test_routes_and_ramps_survive_reset_placement_and_restore():
    lib = H.emu_lib()
    S, n_buses = 64, 5
    bus, gain = _random_routes(np.random.default_rng(4), S, 2, n_buses)
    with _echo_engine(lib, S) as eng, _echo_engine(lib, S) as fresh:
        size = eng.snapshot().size
        eng.set_routes(bus, gain, ramp_frames=500)
        assert eng.snapshot().size == size
        y = eng.mix(_noise(S, 32, 0))
        expect = _reduce(eng, y, SM, n_buses)
        model = Routes(S)
        model.set_routes(bus, gain, ramp_frames=500)
        model.mixed(32)
        _exact(model.buses(y, np.ones(S, bool), n_buses), expect, "model")
        snap = eng.snapshot()
        eng.reset(0, S)
        _exact(expect, _reduce(eng, y, SM, n_buses), "after reset_streams")
        eng.set_placement("auto")
        _exact(expect, _reduce(eng, y, TILED, n_buses), "after AUTO")
        eng.set_placement("caller")
        _exact(expect, _reduce(eng, y, SM, n_buses), "after CALLER")
        eng.restore(fresh.snapshot())
        _exact(expect, _reduce(eng, y, SM, n_buses), "after restore")
        fresh.restore(snap)
        assert fresh.snapshot().size == size


def test_bad_arguments_are_argument_errors_and_change_nothing():
    lib = H.emu_lib()
    S = 40
    bus, gain = _random_routes(np.random.default_rng(6), S, 2, 4)
    with _echo_engine(lib, S) as eng, _echo_engine(lib, S) as twin:
        for e in (eng, twin):
            e.set_routes(bus, gain, ramp_frames=64)
            e.mix(_noise(S, 16, 1))
        b1 = np.zeros((1, 1), np.int32)
        g1 = np.ones((1, 1), F32)
        bad = [
            (-1, 1, 1, b1, g1, 0), (40, 1, 1, b1, g1, 0), (39, 2, 1, np.zeros((2, 1), np.int32), None, 0), (0, 0, 1, b1, g1, 0),
            (0, 1, 0, b1, g1, 0), (0, 1, 5, np.zeros((1, 5), np.int32), None, 0), (0, 1, 1, None, g1, 0),
            (0, 1, 1, np.array([[-2]], np.int32), g1, 0), (0, 1, 2, np.array([[3, 3]], np.int32), None, 0),
            (0, 1, 1, b1, np.array([[np.inf]], F32), 0), (0, 1, 1, b1, np.array([[np.nan]], F32), 0),
            (0, 1, 1, b1, g1, -1), (0, 1, 1, b1, g1, (1 << 24) + 1),
        ]
        for first, n, R, bb, gg, ramp in bad:
            rc = lib.oalsfx_engine_set_routes(eng._h, first, n, R, None if bb is None else bb.ctypes.data,
                                              None if gg is None else gg.ctypes.data, ramp)
            assert rc == -1, (first, n, R, ramp)
        # a bus index above every other keeps n_buses = 4 valid only if refused
        big = np.array([[9]], np.int32)
        assert lib.oalsfx_engine_set_routes(eng._h, 0, 1, 1, big.ctypes.data, None, -5) == -1
        assert lib.oalsfx_engine_set_routes(eng._h, 0, 1, 1, b1.ctypes.data, None, 1 << 24) == 0
        assert lib.oalsfx_engine_set_routes(twin._h, 0, 1, 1, b1.ctypes.data, None, 1 << 24) == 0
        for blk in range(2):
            x = _noise(S, 24, 2 + blk)
            ye, be = _mix_buses(eng, x, 4)
            yt, bt = _mix_buses(twin, x, 4)
            _exact(yt, ye, "dst")
            _exact(bt, be, "buses after refused calls")

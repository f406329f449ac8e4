"""Bus formats and pan routes (oalsfx_engine_set_bus_format / set_route_pans) on the CPU build of the engine (tests/_build):
bit-exact against the numpy model (pan_model.py) on the uint32 images -- mono, stereo and 5.1 engines into buses of another
channel count, pan and scalar routes in one plan, ramps across blocks and kind switches, pauses, both layouts and both
placements -- and every argument error."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from pan_model import Pans
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

SM, TILED = ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED
F32 = np.float32
PAIRS = {"mono-stereo": (F.mono, F.stereo), "stereo-mono": (F.stereo, F.mono), "stereo-5.1": (F.stereo, F.five_point_one),
         "5.1-stereo": (F.five_point_one, F.stereo), "stereo-stereo": (F.stereo, F.stereo)}


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


def _exact(expect, got, what=""):
    assert expect.shape == got.shape, (what, expect.shape, got.shape)
    bad = np.flatnonzero(expect.view(np.uint32) != got.view(np.uint32))
    assert bad.size == 0, (what, "mismatches", bad.size, "first", np.unravel_index(bad[0], expect.shape), H.max_abs_diff(expect, got))


def _reduce(eng, x, layout, n_buses, offset=0):
    """reduce_buses of rows x; with `offset` the block and the bus buffer start `offset` floats into their arrays."""
    frames = x.shape[1]
    xl = _to_layout(x, layout).ravel()
    src = np.concatenate([np.zeros(offset, F32), xl])
    store = np.full(offset + n_buses * frames * eng.bus_channels, F32(3.0))
    eng._check(eng.lib.oalsfx_engine_reduce_buses(eng._h, frames, src.ctypes.data + 4 * offset, layout, n_buses,
                                                  store.ctypes.data + 4 * offset, None))
    return store[offset:].reshape(n_buses, frames, eng.bus_channels)


def _engine(lib, S, fmt, bus_fmt, placement="caller", echo=False):
    eng = ox.Engine(S, fmt, 48000, 1, lib=lib)
    eng.set_placement(placement)
    if echo:
        for p in range(7):
            eng.set_effect(0, T.echo, ox.default_props(T.echo, lib=lib, delay_=0.01 + 0.002 * p), first_stream=p * S // 7,
                           n_streams=(p + 1) * S // 7 - p * S // 7)
    eng.set_bus_format(bus_fmt)
    return eng


def _random_routes(rng, S, R, n_buses, none=0.15):
    bus = np.stack([rng.choice(n_buses, R, replace=False) for _ in range(S)]).astype(np.int32)
    bus[rng.random(bus.shape) < none] = ox.BUS_NONE
    return bus


def _random_pans(rng, shape):
    """Pan matrices of ordinary, zero, negative, tiny and unit coefficients."""
    m = (rng.standard_normal(shape) * 0.8).astype(F32)
    m[rng.random(shape) < 0.15] = F32(0.0)
    m[rng.random(shape) < 0.05] = F32(1e-30)
    m[rng.random(shape) < 0.1] = F32(1.0)
    return m


def _noise(S, C, frames, seed):
    return np.stack([H.noise(seed + s, C, frames) for s in range(S)])


def _mix_buses(eng, x, n_buses, layout=SM):
    S, frames, C = x.shape
    xl = _to_layout(x, layout)
    y = np.full_like(xl, 1.5)
    buses = np.full((n_buses, frames, eng.bus_channels), F32(3.0))
    eng.mix_buses(xl, y, frames, buses, layout=layout)
    if layout == TILED:
        y = y.transpose(0, 3, 1, 2).reshape(-1, frames, C)[:S]
    return np.ascontiguousarray(y), buses


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("pair", list(PAIRS))
def test_pans_match_the_model(pair, layout):
    """150 streams (ragged last tile), 1..4 routes per stream over 12 buses: pan routes on the first streams, scalar routes
    on the rest, in one plan; a zero coefficient of a stream holding an Inf puts NaN on its bus channels, as the model does."""
    lib = H.emu_lib()
    S = 150
    fmt, bus_fmt = PAIRS[pair]
    rng = np.random.default_rng(int(fmt) * 10 + int(bus_fmt) + layout)
    active = np.ones(S, dtype=bool)
    with _engine(lib, S, fmt, bus_fmt) as eng:
        C, Cb = eng.channels, eng.bus_channels
        model = Pans(S, C, Cb)
        for R in (1, 2, 3, 4):
            bus = _random_routes(rng, S, R, 12)
            bus[bus == 5] = ox.BUS_NONE                      # bus 5 is empty
            pans = _random_pans(rng, (S, R, Cb, C))
            gain = (rng.standard_normal((S, R)) * 2).astype(F32)
            half = S // 2 + 3
            eng.set_route_pans(pans[:half], bus[:half])
            model.set_route_pans(pans[:half], bus[:half])
            eng.set_routes(bus[half:], gain[half:], first_stream=half)
            model.set_routes(bus[half:], gain[half:], first_stream=half)
            for frames in (37, 1, 64):
                x = _rows(S, frames, C, 100 * R + frames)
                _exact(model.buses(x, active, 12), _reduce(eng, x, layout, 12), (R, frames))
        if pair == "stereo-stereo":   # swap and balance matrices
            swap = np.array([[0, 1], [1, 0]], F32)
            balance = np.array([[0.25, 0], [0, 1.5]], F32)
            m = np.stack([swap if s % 2 else balance for s in range(S)])
            eng.set_route_pans(m, np.arange(S) % 12)
            model.set_route_pans(m, np.arange(S) % 12)
            x = _rows(S, 40, C, 5)
            got = _reduce(eng, x, layout, 12)
            _exact(model.buses(x, active, 12), got, "swap / balance")
        s = 0
        zero = np.zeros((1, 1, Cb, C), F32)
        eng.set_route_pans(zero, [[4]], first_stream=s)
        model.set_route_pans(zero, [[4]], first_stream=s)
        x = _rows(S, 8, C, 3)
        x[s, 2, 0] = np.inf
        got = _reduce(eng, x, layout, 12)
        _exact(model.buses(x, active, 12), got, "0 * Inf")
        assert np.isnan(got[4, 2]).all()


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_scalar_routes_into_another_format_match_by_index(layout):
    """Default and set_routes routing of a mono engine into stereo buses feeds the left channel only; a 5.1 engine into
    stereo buses feeds its first two channels; a stereo engine into 5.1 buses its first two bus channels."""
    lib = H.emu_lib()
    S = 70
    for fmt, bus_fmt in ((F.mono, F.stereo), (F.five_point_one, F.stereo), (F.stereo, F.five_point_one)):
        with _engine(lib, S, fmt, bus_fmt) as eng, ox.Engine(S, fmt, 48000, 1, lib=lib) as plain:
            C, Cb = eng.channels, eng.bus_channels
            x = _rows(S, 33, C, int(fmt))
            gain = np.random.default_rng(2).standard_normal((S, 1)).astype(F32)
            routing = (np.arange(S) % 3).astype(np.int32)
            for eng_call in ("default", "set_routes"):
                if eng_call == "set_routes":
                    for e in (eng, plain):
                        e.set_routes(routing, gain, ramp_frames=0)
                got = _reduce(eng, x, layout, 3)
                same = _reduce(plain, x, layout, 3)
                m = min(C, Cb)
                _exact(np.ascontiguousarray(same[:, :, :m]), np.ascontiguousarray(got[:, :, :m]), (fmt, bus_fmt, eng_call))
                assert not got[:, :, m:].view(np.uint32).any()
                model = Pans(S, C, Cb)
                if eng_call == "set_routes":
                    model.set_routes(routing, gain)
                _exact(model.buses(x, np.ones(S, bool), 3), got, "model")


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_identity_pans_are_scalar_routes(layout):
    """Cb == C: identity * g gives set_routes(g)'s bits on a finite block, steady and over a ramp; C == Cb == 1: a pan route
    is a scalar route bit for bit, also with Inf and NaN in the block."""
    lib = H.emu_lib()
    S, n_buses = 100, 6
    rng = np.random.default_rng(9)
    bus = _random_routes(rng, S, 2, n_buses)
    gain = (rng.standard_normal((S, 2)) * 2).astype(F32)
    gain[rng.random(gain.shape) < 0.2] = F32(0.0)
    for fmt in (F.stereo, F.five_point_one, F.mono):
        with _engine(lib, S, fmt, fmt, echo=True) as p, _engine(lib, S, fmt, fmt, echo=True) as g:
            C = p.channels
            eye = gain[:, :, None, None] * np.eye(C, dtype=F32)
            for blk, ramp in enumerate((0, 90, 0)):
                p.set_route_pans(eye, bus, ramp_frames=ramp)
                g.set_routes(bus, gain, ramp_frames=ramp)
                x = _noise(S, C, 48, blk)
                yp, bp = _mix_buses(p, x, n_buses, layout)
                yg, bg = _mix_buses(g, x, n_buses, layout)
                _exact(yg, yp, "dst")
                _exact(bg, bp, (fmt, blk, "identity"))
            if fmt == F.mono:
                x = _rows(S, 20, 1, 4)
                x[3, 5, 0], x[7, 2, 0] = np.inf, np.nan
                _exact(_reduce(g, x, layout, n_buses), _reduce(p, x, layout, n_buses), "mono with Inf / NaN")


def test_a_pan_ramp_over_blocks_is_the_model_and_one_long_call():
    """A 300-frame pan ramp from scalar routes over mix_buses blocks of 128 / 64 / 37 frames, alternating layouts; the same
    frames as one call give the same bits."""
    lib = H.emu_lib()
    S, n_buses = 70, 10
    rng = np.random.default_rng(3)
    bus = _random_routes(rng, S, 2, n_buses)
    pans = _random_pans(rng, (S, 2, 2, 1))
    blocks = [128, 64, 37, 128, 64]
    x = _noise(S, 1, sum(blocks), 5)
    with _engine(lib, S, F.mono, F.stereo, echo=True) as eng, _engine(lib, S, F.mono, F.stereo, echo=True) as whole:
        model = Pans(S, 1, 2)
        warm = _noise(S, 1, 16, 99)
        for e in (eng, whole):
            e.set_routes(bus[:, :1], np.full((S, 1), 0.5, F32))
            e.mix(warm)
            e.set_route_pans(pans, bus, ramp_frames=300)
        model.set_routes(bus[:, :1], np.full((S, 1), 0.5, F32))
        model.mixed(16)
        model.set_route_pans(pans, bus, ramp_frames=300)
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


def test_kind_switches_and_mid_ramp_changes():
    """Rows of ones read the coefficients off the bus.  scalar -> pan with a ramp starts from the gain on the diagonal; a pan
    change mid-ramp starts from the coefficients of the last mixed frame; set_routes with a ramp keeps a pan route and ramps
    it to the diagonal; set_routes without a ramp makes it scalar at once; set_route_pans without a ramp applies at once."""
    lib = H.emu_lib()
    S = 4
    with _engine(lib, S, F.stereo, F.stereo) as eng:
        model = Pans(S, 2, 2)
        routing = np.arange(S, dtype=np.int32)
        eng.route(routing)
        model.set_routes(routing)
        rng = np.random.default_rng(5)

        def step(n, what):
            eng.mix(np.zeros((S, n, 2), F32))
            model.mixed(n)
            x = _rows(S, n, 2, n)
            _exact(model.buses(x, np.ones(S, bool), S), _reduce(eng, x, SM, S), what)
            _exact(model.buses(x, np.ones(S, bool), S), _reduce(eng, x, TILED, S), what + " TILED")

        step(10, "start")
        calls = [
            ("pans", 8, "scalar -> pan, ramp"), ("pans", 6, "pan -> pan mid-ramp"), ("gains", 5, "pan -> diagonal, ramp"),
            ("gains", 4, "gain change on a ramping pan route"), ("gains", 0, "pan -> scalar at once"),
            ("pans", 0, "scalar -> pan at once"), ("gains", 3, "pan -> diagonal again"),
        ]
        for kind, ramp, what in calls:
            if kind == "pans":
                m = _random_pans(rng, (2, 1, 2, 2))
                eng.set_route_pans(m, routing[1:3], first_stream=1, ramp_frames=ramp)
                model.set_route_pans(m, routing[1:3], first_stream=1, ramp_frames=ramp)
            else:
                g = rng.standard_normal((2, 1)).astype(F32)
                eng.set_routes(routing[1:3], g, first_stream=1, ramp_frames=ramp)
                model.set_routes(routing[1:3], g, first_stream=1, ramp_frames=ramp)
            step(3, what)
            step(4, what + ", next block")
        # a new pan route fades in from 0 next to an existing one
        m = _random_pans(rng, (1, 2, 2, 2))
        eng.set_route_pans(m, [[0, 3]], first_stream=0, ramp_frames=7)
        model.set_route_pans(m, [[0, 3]], first_stream=0, ramp_frames=7)
        step(5, "fade-in of a new pan route")


@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_paused_streams_are_not_members(placement):
    """Streams pause and resume during a pan ramp: the buses are the model over the active streams for both placements;
    paused rows are never read (NaN there would show)."""
    lib = H.emu_lib()
    S, n_buses = 90, 7
    rng = np.random.default_rng(11)
    bus = _random_routes(rng, S, 2, n_buses)
    pans = _random_pans(rng, (S, 2, 6, 2))
    with _engine(lib, S, F.stereo, F.five_point_one, placement, echo=True) as eng, \
            _engine(lib, S, F.stereo, F.five_point_one, "caller", echo=True) as ref:
        model = Pans(S, 2, 6)
        active = np.ones(S, dtype=bool)
        for e in (eng, ref):
            e.set_route_pans(pans, bus, ramp_frames=200)
        model.set_route_pans(pans, bus, ramp_frames=200)
        for blk in range(5):
            if blk > 0:
                flip = rng.choice(S, 15, replace=False)
                active[flip] = ~active[flip]
                for e in (eng, ref):
                    for s in flip:
                        e.set_active(bool(active[s]), int(s), 1)
            x = _noise(S, 2, 48, 30 + blk)
            y, buses = _mix_buses(eng, x, n_buses, TILED if blk % 2 else SM)
            _, ref_buses = _mix_buses(ref, x, n_buses)
            model.mixed(48)
            _exact(model.buses(y, active, n_buses), buses, blk)
            _exact(ref_buses, buses, ("CALLER vs", placement))
            junk = y.copy()
            junk[~active] = np.nan
            _exact(buses, _reduce(eng, junk, SM, n_buses), "paused rows read")


@pytest.mark.parametrize("layout", [SM, TILED], ids=["stream_major", "tiled"])
def test_odd_long_and_unaligned_calls(layout):
    """5000 frames (three chunks), 37 and 3 frames, and a block and bus buffer one float off their 16-byte alignment."""
    lib = H.emu_lib()
    S, n_buses = 140, 9
    rng = np.random.default_rng(21)
    for fmt, bus_fmt in ((F.mono, F.stereo), (F.stereo, F.five_point_one)):
        with _engine(lib, S, fmt, bus_fmt) as eng:
            C, Cb = eng.channels, eng.bus_channels
            bus = _random_routes(rng, S, 2, n_buses)
            pans = _random_pans(rng, (S, 2, Cb, C))
            model = Pans(S, C, Cb)
            eng.mix(np.zeros((S, 64, C), F32))
            model.mixed(64)
            eng.set_route_pans(pans, bus, ramp_frames=2600)
            model.set_route_pans(pans, bus, ramp_frames=2600)
            for frames, offset in ((5000, 0), (37, 1), (3, 0), (64, 1)):
                x = _rows(S, frames, C, frames)
                expect = model.buses(x, np.ones(S, bool), n_buses)
                _exact(expect, _reduce(eng, x, layout, n_buses, offset), (fmt, frames, offset))


def test_format_and_pans_survive_reset_placement_and_restore():
    lib = H.emu_lib()
    S, n_buses = 64, 5
    rng = np.random.default_rng(4)
    bus = _random_routes(rng, S, 2, n_buses)
    pans = _random_pans(rng, (S, 2, 2, 1))
    with _engine(lib, S, F.mono, F.stereo, echo=True) as eng, _engine(lib, S, F.mono, F.mono, echo=True) as fresh:
        size = eng.snapshot().size
        before = eng.device_bytes
        eng.set_route_pans(pans, bus, ramp_frames=500)
        assert eng.snapshot().size == size
        y = eng.mix(_noise(S, 1, 32, 0))
        expect = _reduce(eng, y, SM, n_buses)
        assert eng.device_bytes > before
        model = Pans(S, 1, 2)
        model.set_route_pans(pans, bus, ramp_frames=500)
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
        assert eng.bus_channels == 2
        fresh.restore(snap)
        assert fresh.snapshot().size == size


def test_mix_buses_refuses_before_it_mixes():
    """A mix_buses refused for n_buses advances neither the streams nor the frame clock: the next blocks match a twin that
    never saw the call, during a pan ramp."""
    lib = H.emu_lib()
    S, n_buses = 40, 4
    rng = np.random.default_rng(6)
    bus = _random_routes(rng, S, 2, n_buses)
    pans = _random_pans(rng, (S, 2, 2, 1))
    with _engine(lib, S, F.mono, F.stereo, echo=True) as eng, _engine(lib, S, F.mono, F.stereo, echo=True) as twin:
        for e in (eng, twin):
            e.set_route_pans(pans, bus, ramp_frames=100)
            _mix_buses(e, _noise(S, 1, 16, 1), n_buses)
        x = _noise(S, 1, 24, 2)
        y = np.empty_like(x)
        small = np.zeros((1, 24, 2), F32)
        rc = lib.oalsfx_engine_mix_buses(eng._h, 24, x.ctypes.data, y.ctypes.data, SM, 1, small.ctypes.data, None)
        assert rc == -1
        for blk in range(2):
            x = _noise(S, 1, 24, 3 + blk)
            ye, be = _mix_buses(eng, x, n_buses)
            yt, bt = _mix_buses(twin, x, n_buses)
            _exact(yt, ye, "dst")
            _exact(bt, be, "buses after a refused mix_buses")


def test_bad_arguments_are_errors_and_change_nothing():
    lib = H.emu_lib()
    S = 40
    rng = np.random.default_rng(6)
    bus = _random_routes(rng, S, 2, 4)
    pans = _random_pans(rng, (S, 2, 6, 2))
    with _engine(lib, S, F.stereo, F.five_point_one, echo=True) as eng, \
            _engine(lib, S, F.stereo, F.five_point_one, echo=True) as twin:
        for e in (eng, twin):
            e.set_route_pans(pans, bus, ramp_frames=64)
            e.mix(_noise(S, 2, 16, 1))
        for fmt in (0, 8, -1):
            assert lib.oalsfx_engine_set_bus_format(eng._h, fmt) == -2, fmt
        assert lib.oalsfx_engine_set_bus_format(eng._h, int(F.stereo)) == -1        # pan routes are sized for Cb = 6
        assert lib.oalsfx_engine_set_bus_format(eng._h, int(F.five_point_one)) == 0  # the current format again
        assert lib.oalsfx_engine_set_bus_format(eng._h, int(F.five_point_one_rear)) == 0   # the same Cb
        assert lib.oalsfx_engine_set_bus_format(twin._h, int(F.five_point_one_rear)) == 0
        b1 = np.zeros((1, 1), np.int32)
        m1 = np.ones((1, 1, 6, 2), F32)
        inf = m1.copy()
        inf[0, 0, 3, 1] = np.inf
        nan = m1.copy()
        nan[0, 0, 0, 0] = np.nan
        bad = [
            (-1, 1, 1, b1, m1, 0), (40, 1, 1, b1, m1, 0), (39, 2, 1, np.zeros((2, 1), np.int32), np.ones((2, 1, 6, 2), F32), 0),
            (0, 0, 1, b1, m1, 0), (0, 1, 0, b1, m1, 0), (0, 1, 5, np.zeros((1, 5), np.int32), np.ones((1, 5, 6, 2), F32), 0),
            (0, 1, 1, None, m1, 0), (0, 1, 1, b1, None, 0), (0, 1, 1, np.array([[-2]], np.int32), m1, 0),
            (0, 1, 2, np.array([[3, 3]], np.int32), np.ones((1, 2, 6, 2), F32), 0), (0, 1, 1, b1, inf, 0), (0, 1, 1, b1, nan, 0),
            (0, 1, 1, b1, m1, -1), (0, 1, 1, b1, m1, (1 << 24) + 1), (0, 1, 1, np.array([[9]], np.int32), m1, -5),
        ]
        for first, n, R, bb, mm, ramp in bad:
            rc = lib.oalsfx_engine_set_route_pans(eng._h, first, n, R, None if bb is None else bb.ctypes.data,
                                                  None if mm is None else mm.ctypes.data, ramp)
            assert rc == -1, (first, n, R, ramp)
        assert lib.oalsfx_engine_set_route_pans(None, 0, 1, 1, b1.ctypes.data, m1.ctypes.data, 0) == -1
        assert lib.oalsfx_engine_set_bus_format(None, int(F.stereo)) == -1
        for blk in range(2):
            x = _noise(S, 2, 24, 2 + blk)
            ye, be = _mix_buses(eng, x, 4)
            yt, bt = _mix_buses(twin, x, 4)
            _exact(yt, ye, "dst")
            _exact(bt, be, "buses after refused calls")
        # once no route is a pan route, the channel count may change
        eng.set_routes(bus, np.ones(bus.shape, F32))
        eng.set_bus_format(F.stereo)
        assert eng.bus_channels == 2


def test_pan_image_grows_with_the_plan():
    """The plan grows while no route has a matrix -- paused streams resume, streams gain routes -- and then a pan change
    that keeps the (stream, bus) pairs writes one entry: the pan image covers the whole plan, and the buses stay the
    model's."""
    lib = H.emu_lib()
    S, n_buses = 100, 6
    rng = np.random.default_rng(17)
    with _engine(lib, S, F.mono, F.stereo) as eng:
        model = Pans(S, 1, 2)
        active = np.ones(S, dtype=bool)
        routing = (np.arange(S) % n_buses).astype(np.int32)

        def check(what):
            x = _rows(S, 24, 1, len(what))
            for layout in (SM, TILED):
                _exact(model.buses(x, active, n_buses), _reduce(eng, x, layout, n_buses), (what, layout))

        eng.set_active(False, 50, 50)
        active[50:] = False
        pans = _random_pans(rng, (50, 2, 1))
        eng.set_route_pans(pans, routing[:50])
        model.set_route_pans(pans, routing[:50])
        check("pans on the active half")
        eng.route(routing)
        model.set_routes(routing)
        check("scalar routes again")
        eng.set_active(True, 50, 50)
        active[50:] = True
        check("all streams active")
        m = _random_pans(rng, (1, 2, 1))
        eng.set_route_pans(m, routing[:1])
        model.set_route_pans(m, routing[:1])
        check("one pan route in the grown plan")
        two = np.stack([routing, (routing + 1) % n_buses], axis=1)
        eng.route(routing)
        model.set_routes(routing)
        eng.set_routes(two, np.full(two.shape, 0.5, F32))
        model.set_routes(two, np.full(two.shape, 0.5, F32))
        check("two scalar routes per stream")
        m = _random_pans(rng, (1, 2, 2, 1))
        eng.set_route_pans(m, two[S - 1:], first_stream=S - 1, ramp_frames=30)
        model.set_route_pans(m, two[S - 1:], first_stream=S - 1, ramp_frames=30)
        check("pan routes on the last stream of a plan twice as long")

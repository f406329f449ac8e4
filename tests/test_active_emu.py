"""Paused streams and stream resets (oalsfx_engine_set_active / oalsfx_engine_reset_streams) on the CPU build of the
engine (tests/_build): a paused stream is a reference Api whose mix is not called, its rows are zeros, and a reset
stream continues like a fresh Api with the same configuration.  Bit-exact against the CPU checker."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

N_PRESETS = 13
FILL = np.float32(1.5)   # dst is pre-filled with this: a paused row must be overwritten with +0.0f


def _echo(lib, p):
    return ox.default_props(T.echo, lib=lib, delay_=0.01 + 0.003 * p, feedback_=0.2 + 0.01 * p)


def _input_block(S, frames, seed, layout):
    x = np.stack([H.noise(seed + s, 2, frames) for s in range(S)])      # [S][F][C]
    if layout == ox.LAYOUT_STREAM_MAJOR:
        return x, x
    T_ = (S + 31) // 32
    t = np.zeros((T_ * 32, frames, 2), dtype=np.float32)
    t[:S] = x
    return x, np.ascontiguousarray(t.reshape(T_, 32, frames, 2).transpose(0, 2, 3, 1))


def _rows(y, S, layout):
    if layout == ox.LAYOUT_STREAM_MAJOR:
        return y
    T_, frames = y.shape[0], y.shape[1]
    return y.transpose(0, 3, 1, 2).reshape(T_ * 32, frames, 2)[:S]


class _Voices:
    """One engine and, per stream, the reference script of what that stream's Api saw: its configuration calls and a
    ("mix", n) for every block it was mixed in, with the inputs of those blocks."""

    def __init__(self, lib, S, slots, placement):
        self.lib, self.S = lib, S
        self.eng = ox.Engine(S, F.stereo, 48000, len(slots), lib=lib)
        if placement == "auto":
            self.eng.set_placement("auto")
        self.slots = len(slots)
        self.script = [[] for _ in range(S)]
        self.inputs = [[] for _ in range(S)]
        self.outputs = [[] for _ in range(S)]
        self.active = np.ones(S, dtype=bool)
        self.config = [[None] * (self.slots + 1) for _ in range(S)]
        self.pending = np.zeros(S, dtype=np.int64)
        for s in range(S):
            for slot, (t, p) in enumerate(slots):
                self.set_effect(s, slot, t, p)
            self.script[s].append(("apply",))

    def close(self):
        self.eng.close()

    def set_effect(self, s, slot, t, p, apply=False):
        self.eng.set_effect(slot, t, p, first_stream=s, n_streams=1)
        self.script[s] += [("type", slot, t)] + ([("props", slot, p)] if p is not None else []) + ([("apply",)] if apply else [])
        self.config[s][slot] = (int(t), None if p is None else bytes(p))
        self.pending[s] |= 1 << slot

    def set_filtered_sends(self, s):
        self.eng.set_sends(direct=(0.8, 0.5, 1.0), aux=[(1.0, 0.25, 1.0)] * self.slots, first_stream=s, n_streams=1)
        self.script[s] += [("send", -1, (0.8, 0.5, 1.0))] + [("send", i, (1.0, 0.25, 1.0)) for i in range(self.slots)]
        self.config[s][self.slots] = "filtered"

    def set_active(self, s, on):
        self.eng.set_active(on, first_stream=s, n_streams=1)
        self.active[s] = on

    def key(self, s):
        return (tuple(map(str, self.config[s])), int(self.pending[s]))

    def mix(self, frames, seed, layout, space):
        x, xin = _input_block(self.S, frames, seed, layout)
        y = np.full_like(xin, FILL)
        self.eng.mix(xin, y, frames=frames, layout=layout, space=space)
        rows = _rows(y, self.S, layout)
        for s in range(self.S):
            if self.active[s]:
                self.script[s].append(("mix", frames))
                self.inputs[s].append(x[s])
                self.outputs[s].append(rows[s].copy())
                self.pending[s] = 0
        return rows

    def check_against(self, checker, streams=None):
        for s in (range(self.S) if streams is None else streams):
            if not self.inputs[s]:
                continue
            expect = H.run_script_orc(checker, F.stereo, 48000, self.slots, self.script[s], np.concatenate(self.inputs[s]))
            got = np.concatenate(self.outputs[s])
            assert np.array_equal(expect.view(np.uint32), got.view(np.uint32)), (s, H.max_abs_diff(expect, got))


def _states(eng, streams, slots):
    return {s: [eng.debug_state(s, slot) for slot in range(slots)] for s in streams}


@pytest.mark.parametrize("space", [ox.SPACE_HOST, ox.SPACE_DEVICE], ids=["host", "device"])
@pytest.mark.parametrize("layout", [ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED], ids=["stream_major", "tiled"])
@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_paused_streams_are_apis_whose_mix_is_not_called(checker, placement, layout, space):
    """77 streams (ragged last tile), echo with 13 presets and chorus -> flanger, shelf-filtered sends on some streams.
    Before every block about 40 % of the streams pause and the others resume; preset and type changes also hit paused
    streams.  Every stream's output over the blocks it was mixed in equals its checker Api fed only those blocks, every
    paused row is +0.0f, a paused stream's state does not move, and (AUTO) no launched tile mixes active and paused."""
    lib = H.emu_lib()
    S = 77
    rng = np.random.default_rng(11)
    v = _Voices(lib, S, [(T.echo, None), (T.chorus, None)], placement)
    try:
        for s in range(S):
            v.set_effect(s, 0, T.echo, _echo(lib, s % N_PRESETS), apply=False)
            if s % 9 == 4:
                v.set_filtered_sends(s)
            v.script[s].append(("apply",))
        for b, frames in enumerate([64, 48, 1, 64, 37, 64]):
            for s in range(S):
                v.set_active(s, bool(rng.random() >= 0.4))
            if b > 0:
                for s in rng.choice(S, 8, replace=False):
                    v.set_effect(int(s), 0, T.echo, _echo(lib, int(rng.integers(0, N_PRESETS + 3))), apply=True)
                for s in rng.choice(S, 4, replace=False):
                    v.set_effect(int(s), 1, T.flanger, ox.default_props(T.flanger, lib=lib, rate_=0.2 + 0.05 * int(rng.integers(0, 2))),
                                 apply=True)
            assert (~v.active).sum() > 0 and v.active.sum() > 0
            keys = [v.key(s) for s in range(S)]
            paused = [s for s in range(S) if not v.active[s]]
            before = _states(v.eng, paused, 2)
            rows = v.mix(frames, 1000 * b, layout, space)
            assert not rows[~v.active].view(np.uint32).any(), f"block {b}: a paused row is not +0.0f"
            assert _states(v.eng, paused, 2) == before, f"block {b}: a paused stream's state moved"
            if placement == "auto":
                lanes, _ = v.eng.lanes()
                by_tile = {}
                for s in range(S):
                    by_tile.setdefault(int(lanes[s]) // 32, []).append(s)
                for members in by_tile.values():
                    live = [s for s in members if v.active[s]]
                    if live:
                        assert len(live) == len(members), f"block {b}: a tile mixes active and paused streams"
                        assert len({keys[s] for s in live}) == 1, f"block {b}: a launched tile holds two keys"
        v.check_against(checker)
    finally:
        v.close()


@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_everything_paused_launches_nothing_and_keeps_the_state(placement):
    lib = H.emu_lib()
    S = 50
    with ox.Engine(S, F.stereo, 48000, 2, lib=lib) as eng:
        if placement == "auto":
            eng.set_placement("auto")
        for s in range(S):
            eng.set_effect(0, T.echo, _echo(lib, s % 3), first_stream=s, n_streams=1)
        eng.set_effect(1, T.eax_reverb)
        eng.mix(np.stack([H.noise(s, 2, 40) for s in range(S)]))
        eng.set_active(False)
        snap, launches = eng.snapshot(), eng.launch_count
        for layout in (ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED):
            _, x = _input_block(S, 33, 7, layout)
            y = np.full_like(x, FILL)
            eng.mix(x, y, frames=33, layout=layout)
            assert not y.view(np.uint32).any()
        assert eng.launch_count == launches
        assert np.array_equal(eng.snapshot(), snap)


@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_set_active_on_every_stream_changes_nothing(placement):
    """Activity flags that are all set select the same kernels, with the same launch count, and give the same bits."""
    lib = H.emu_lib()
    S = 70
    engines = [ox.Engine(S, F.stereo, 48000, 2, lib=lib) for _ in range(2)]
    try:
        for i, eng in enumerate(engines):
            if placement == "auto":
                eng.set_placement("auto")
            if i == 1:
                eng.set_active(True)
            for s in range(S):
                eng.set_effect(0, T.echo, _echo(lib, s % 4), first_stream=s, n_streams=1)
            eng.set_effect(1, T.chorus)
            eng.set_sends(direct=(0.8, 0.5, 1.0), aux=[(1.0, 1.0, 1.0)] * 2, first_stream=5, n_streams=3)
        for b, frames in enumerate([64, 1, 48]):
            if b == 1:
                engines[1].set_active(True, first_stream=0, n_streams=40)
                for eng in engines:
                    eng.set_effect(1, T.flanger, first_stream=10, n_streams=20)
            x = np.stack([H.noise(50 + s, 2, frames) for s in range(S)])
            y0, y1 = engines[0].mix(x), engines[1].mix(x)
            assert np.array_equal(y0.view(np.uint32), y1.view(np.uint32)), b
            assert engines[0].launch_count == engines[1].launch_count
            assert engines[0].last_kernel == engines[1].last_kernel
    finally:
        for eng in engines:
            eng.close()


@pytest.mark.parametrize("placement", ["caller", "auto"])
def test_reset_streams_restart_like_fresh_apis(checker, placement):
    """Echo + EAX reverb on 40 streams; after the second block streams reset: one paused at the time (resumed later),
    one whose reverb is inside a tap cross-fade, a range across a tile boundary.  Each stream equals its old checker Api
    up to the reset and a fresh one with the same configuration after it; right after the reset its integer state equals
    that of a freshly created engine."""
    lib = H.emu_lib()
    S = 40
    reverb = lambda d: ox.default_props(T.eax_reverb, lib=lib, reflections_delay_=0.01 + 0.005 * d, decay_time_=1.0 + 0.2 * d)
    v = _Voices(lib, S, [(T.echo, None), (T.eax_reverb, None)], placement)
    try:
        for s in range(S):
            v.set_effect(s, 0, T.echo, _echo(lib, s % 5))
            v.set_effect(s, 1, T.eax_reverb, reverb(s % 2), apply=True)
        paused_at_reset, fading, span = 17, 33, list(range(28, 36))
        resets = [3, paused_at_reset] + span
        v.mix(64, 0, ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
        v.set_active(paused_at_reset, False)
        v.set_effect(fading, 1, T.eax_reverb, reverb(3), apply=True)       # taps change: a 128-frame cross-fade starts
        v.mix(64, 1, ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
        assert 0 < v.eng.debug_state(fading, 1)["fade_count"] < 128
        for s in [3, paused_at_reset]:
            v.eng.reset(first_stream=s, n_streams=1)
        v.eng.reset(first_stream=span[0], n_streams=len(span))
        assert not v.active[paused_at_reset]
        with ox.Engine(S, F.stereo, 48000, 2, lib=lib) as twin:
            for s in resets:
                twin.set_effect(0, T.echo, _echo(lib, s % 5), first_stream=s, n_streams=1)
                twin.set_effect(1, T.eax_reverb, reverb(3 if s == fading else s % 2), first_stream=s, n_streams=1)
            assert _states(v.eng, resets, 2) == _states(twin, resets, 2)
        # the reset streams' references start over: everything mixed so far belongs to the old Api
        old = {s: (v.script[s], v.inputs[s], v.outputs[s]) for s in resets}
        for s in resets:
            v.script[s] = [("type", 0, T.echo), ("props", 0, _echo(lib, s % 5)),
                           ("type", 1, T.eax_reverb), ("props", 1, reverb(3 if s == fading else s % 2)), ("apply",)]
            v.inputs[s], v.outputs[s] = [], []
            v.pending[s] = 3
        for b, frames in enumerate([50, 64, 64], start=2):
            if b == 3:
                v.set_active(paused_at_reset, True)
            v.mix(frames, 10 * b, ox.LAYOUT_TILED, ox.SPACE_DEVICE)
        assert v.inputs[paused_at_reset] and v.inputs[fading]
        v.check_against(checker)
        for s, (script, inputs, outputs) in old.items():
            if inputs:
                expect = H.run_script_orc(checker, F.stereo, 48000, 2, script, np.concatenate(inputs))
                assert np.array_equal(expect.view(np.uint32), np.concatenate(outputs).view(np.uint32)), s
    finally:
        v.close()


def test_bad_ranges_are_argument_errors():
    lib = H.emu_lib()
    with ox.Engine(40, F.stereo, 48000, 1, lib=lib) as eng:
        for call in (lambda f, n: eng.set_active(False, f, n), lambda f, n: eng.reset(f, n)):
            for f, n in ((-1, 1), (0, 0), (39, 2), (0, -3), (40, 1)):
                with pytest.raises(ox.OalsfxError) as err:
                    call(f, n)
                assert err.value.code == -1

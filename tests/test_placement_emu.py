"""Stream placement inside the engine (OALSFX_PLACEMENT_AUTO) on the CPU build of the engine (tests/_build, the host
logic and kernel bodies compiled for the CPU): the planner's invariants after every block of a randomized script,
outputs bit-identical to an unplaced engine on every caller stream, and snapshots in caller stream order."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

N_PRESETS = 13


def _echo(lib, p):
    return ox.default_props(T.echo, lib=lib, delay_=0.01 + 0.003 * p, feedback_=0.2 + 0.01 * p)


class _Twins:
    """The same history on an unplaced engine and on one in AUTO mode, plus the caller-side view of every stream's
    settings (label) and pending-update bits, which together are the placement key."""

    def __init__(self, lib, streams, auto=True):
        self.lib, self.S = lib, streams
        self.ref = ox.Engine(streams, F.stereo, 48000, 2, lib=lib)
        self.eng = ox.Engine(streams, F.stereo, 48000, 2, lib=lib)
        if auto:
            self.eng.set_placement("auto")
        self.config = [[("echo", s % N_PRESETS), ("chorus", 0), (1.0, 1.0, 1.0)] for s in range(streams)]
        self.pending = np.zeros(streams, dtype=np.int64)
        for s in range(streams):
            self._apply_effect(s, 0)
            self._apply_effect(s, 1)

    def close(self):
        self.ref.close()
        self.eng.close()

    def _apply_effect(self, s, slot):
        kind, p = self.config[s][slot]
        if kind == "echo":
            args = (T.echo, _echo(self.lib, p))
        elif kind == "chorus":
            args = (T.chorus, None)
        else:
            args = (T.flanger, ox.default_props(T.flanger, lib=self.lib, rate_=0.2 + 0.05 * p))
        for e in (self.ref, self.eng):
            e.set_effect(slot, *args, first_stream=s, n_streams=1)
        self.pending[s] |= 1 << slot

    def preset(self, s, p):
        self.config[s][0] = ("echo", p)
        self._apply_effect(s, 0)

    def flanger(self, s, p):
        self.config[s][1] = ("flanger", p)
        self._apply_effect(s, 1)

    def sends(self, s, g):
        self.config[s][2] = g
        for e in (self.ref, self.eng):
            e.set_sends(direct=g, aux=[(1.0, 1.0, 1.0)] * 2, first_stream=s, n_streams=1)

    def keys(self):
        return [(tuple(map(tuple, [c[0], c[1], c[2]])), int(self.pending[s])) for s, c in enumerate(self.config)]

    def mix(self, x, layout, space):
        y_ref, y = np.zeros_like(x), np.zeros_like(x)
        frames = x.shape[1] if layout == ox.LAYOUT_STREAM_MAJOR else x.shape[1]
        self.ref.mix(x, y_ref, frames=frames, layout=layout, space=space)
        self.eng.mix(x, y, frames=frames, layout=layout, space=space)
        self.pending[:] = 0
        return y_ref, y


def _tiles_of(lanes):
    return lanes // 32


def _check_invariants(keys, lanes, count, prev):
    """Planner invariants 1-4 after a placement; `prev` = (lanes, count, keys) before it, or None."""
    S = len(keys)
    assert count % 32 == 0 and lanes.min() >= 0 and lanes.max() < count
    assert len(set(lanes.tolist())) == S, "lane_of_stream is not a permutation"
    tiles = _tiles_of(lanes)
    by_tile = {}
    for s in range(S):
        by_tile.setdefault(int(tiles[s]), set()).add(keys[s])
    assert all(len(v) == 1 for v in by_tile.values()), "a tile holds more than one key"        # 1
    per_key = {}
    members = {}
    for s in range(S):
        per_key.setdefault(keys[s], set()).add(int(tiles[s]))
        members[keys[s]] = members.get(keys[s], 0) + 1
    for k, ts in per_key.items():
        assert len(ts) <= (members[k] + 31) // 32 + 1, ("too many tiles for a key", len(ts), members[k])  # 3
    if prev is None:
        return
    plane, pcount, pkeys = prev
    assert count >= pcount                                                                     # 4: never shrinks
    if count > pcount:                                                                         # 4: reuse first
        assert set(range(pcount // 32)) <= set(by_tile), "the engine grew while a tile was free"
    ptiles = _tiles_of(plane)
    changed = {s for s in range(S) if keys[s] != pkeys[s]}
    pure_before = {}
    for s in range(S):
        pure_before.setdefault(int(ptiles[s]), set()).add(pkeys[s])
    moved = [s for s in range(S) if lanes[s] != plane[s]]
    repacked = {k for k, ts in per_key.items() if len(ts) == (members[k] + 31) // 32}
    for s in moved:                                                                            # 2
        untouched = s not in changed and len(pure_before[int(ptiles[s])]) == 1 and \
            all(keys[t] == pkeys[t] for t in range(S) if ptiles[t] == ptiles[s])
        assert not untouched or keys[s] in repacked, ("a stream in a pure, unchanged tile moved", s)
    outside_repack = [s for s in moved if keys[s] not in repacked]
    assert len(outside_repack) <= len(changed), (len(outside_repack), len(changed))


def _input(S, frames, seed, layout):
    x = np.stack([H.noise(seed + s, 2, frames) for s in range(S)])      # [S][F][C]
    if layout == ox.LAYOUT_STREAM_MAJOR:
        return x
    T_ = (S + 31) // 32
    t = np.zeros((T_ * 32, frames, 2), dtype=np.float32)
    t[:S] = x
    return np.ascontiguousarray(t.reshape(T_, 32, frames, 2).transpose(0, 2, 3, 1))


def _rows(y, S, layout):
    if layout == ox.LAYOUT_STREAM_MAJOR:
        return y
    T_, frames = y.shape[0], y.shape[1]
    return y.transpose(0, 3, 1, 2).reshape(T_ * 32, frames, 2)[:S]


@pytest.mark.parametrize("space", [ox.SPACE_HOST, ox.SPACE_DEVICE], ids=["host", "device"])
@pytest.mark.parametrize("layout", [ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED], ids=["stream_major", "tiled"])
def test_placed_engine_keeps_tiles_pure_and_matches_an_unplaced_one(layout, space):
    """77 streams (ragged last tile), 13 presets in no particular order, a randomized script of preset changes on
    scattered streams, chorus -> flanger type changes and send changes, including a 1-frame block.  After every
    block the placement satisfies invariants 1-4, and every caller stream's output equals the unplaced engine's."""
    lib = H.emu_lib()
    S = 77
    rng = np.random.default_rng(5)
    tw = _Twins(lib, S)
    try:
        prev = None
        for b, frames in enumerate([64, 48, 1, 64, 37, 64, 64]):
            if b > 0:
                for s in rng.choice(S, 6, replace=False):
                    tw.preset(int(s), int(rng.integers(0, N_PRESETS + 3)))
                for s in rng.choice(S, 3, replace=False):
                    tw.flanger(int(s), int(rng.integers(0, 2)))
                for s in rng.choice(S, 2, replace=False):
                    tw.sends(int(s), (0.5 + 0.25 * int(rng.integers(0, 2)), 1.0, 1.0))
            keys = tw.keys()
            x = _input(S, frames, 100 * b, layout)
            y_ref, y = tw.mix(x, layout, space)
            assert np.array_equal(_rows(y_ref, S, layout).view(np.uint32), _rows(y, S, layout).view(np.uint32)), f"block {b}"
            lanes, count = tw.eng.lanes()
            _check_invariants(keys, lanes, count, prev)
            prev = (lanes, count, keys)
        for s in range(0, S, 7):
            for slot in range(2):
                assert tw.eng.debug_state(s, slot) == tw.ref.debug_state(s, slot)
        assert tw.ref.lanes()[0].tolist() == list(range(S))
    finally:
        tw.close()


def test_switching_back_to_caller_placement_restores_identity_lanes():
    lib = H.emu_lib()
    S = 45
    tw = _Twins(lib, S)
    try:
        for b in range(2):
            y_ref, y = tw.mix(_input(S, 40, 10 * b, ox.LAYOUT_STREAM_MAJOR), ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
            assert np.array_equal(y_ref.view(np.uint32), y.view(np.uint32))
        assert tw.eng.lane_of_stream.tolist() != list(range(S))
        tw.eng.set_placement("caller")
        lanes, count = tw.eng.lanes()
        assert lanes.tolist() == list(range(S)) and count == 64
        for b in range(2, 4):
            y_ref, y = tw.mix(_input(S, 40, 10 * b, ox.LAYOUT_STREAM_MAJOR), ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
            assert np.array_equal(y_ref.view(np.uint32), y.view(np.uint32))
            assert tw.eng.last_kernel == tw.ref.last_kernel
        with pytest.raises(ValueError):
            tw.eng.set_placement("sorted")
    finally:
        tw.close()


def test_placed_snapshots_are_in_caller_order_and_restore_across_modes():
    """64 streams: a placed engine's snapshot equals the unplaced engine's byte for byte; it restores into an unplaced
    engine (and the unplaced one's into a placed engine) and both continue bit-exact."""
    lib = H.emu_lib()
    S = 64
    tw = _Twins(lib, S)
    try:
        for b in range(3):
            if b == 1:
                for s in (3, 17, 40, 41):
                    tw.preset(s, 11)
                tw.flanger(9, 1)
            tw.mix(_input(S, 50, 7 * b, ox.LAYOUT_STREAM_MAJOR), ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
        tw.preset(20, 2)   # an update still pending: its bytes are per caller stream
        assert tw.eng.lane_of_stream.tolist() != list(range(S))
        snap_ref, snap = tw.ref.snapshot(), tw.eng.snapshot()
        assert np.array_equal(snap_ref, snap)
        # fresh engines with the same configuration, the other way round
        fresh = _Twins(lib, S, auto=False)
        try:
            fresh.eng.set_placement("auto")
            for s in range(S):
                fresh.config[s] = list(tw.config[s])
                for slot in range(2):
                    fresh._apply_effect(s, slot)
                if tw.config[s][2] != (1.0, 1.0, 1.0):
                    fresh.sends(s, tw.config[s][2])
            fresh.ref.restore(snap)        # placed snapshot -> unplaced engine
            fresh.eng.restore(snap_ref)    # unplaced snapshot -> placed engine
            for b in range(3, 5):
                x = _input(S, 50, 7 * b, ox.LAYOUT_STREAM_MAJOR)
                y_orig, y_orig_placed = tw.mix(x, ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
                y_ref, y = fresh.mix(x, ox.LAYOUT_STREAM_MAJOR, ox.SPACE_HOST)
                for got in (y_orig_placed, y_ref, y):
                    assert np.array_equal(y_orig.view(np.uint32), got.view(np.uint32)), b
            assert np.array_equal(fresh.eng.snapshot(), tw.ref.snapshot())
        finally:
            fresh.close()
    finally:
        tw.close()

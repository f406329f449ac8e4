"""Paused streams and stream resets on the GPU: pausing keeps the fused launches of the active streams (one
class-per-tile launch under AUTO placement, the same kernel as a smaller engine when whole tiles pause under CALLER
placement, the span kernel), paused rows are +0.0f, and sampled streams are bit-exact against the CPU checker fed only
the blocks they were mixed in."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

CHAIN = [T.equalizer, T.chorus, T.echo, T.eax_reverb]


def _assert_exact(expect, got, what=""):
    assert expect.shape == got.shape, (what, expect.shape, got.shape)
    e32 = np.ascontiguousarray(expect, dtype=np.float32).view(np.uint32)
    g32 = np.ascontiguousarray(got, dtype=np.float32).view(np.uint32)
    differ = (e32 != g32) & ~(np.isnan(expect) & np.isnan(got))
    if differ.any():
        bad = np.argwhere(differ)
        raise AssertionError((what, "first mismatch at", tuple(bad[0]), "count", len(bad), "max abs diff", H.max_abs_diff(expect, got)))


def _to_tiled(x):
    S, n, C = x.shape
    return x.reshape(S // 32, 32, n, C).permute(0, 2, 3, 1).contiguous()


def _from_tiled(t):
    T_, n, C, _ = t.shape
    return t.permute(0, 3, 1, 2).reshape(T_ * 32, n, C)


class _Streams:
    """Per sampled stream: the reference script of its Api (configuration calls, a mix per block it was mixed in) and
    the inputs / outputs of those blocks."""

    def __init__(self, sample, fmt, slots):
        self.fmt, self.slots = fmt, slots
        self.script = {s: [] for s in sample}
        self.x = {s: [] for s in sample}
        self.y = {s: [] for s in sample}

    def op(self, s, *ops):
        if s in self.script:
            self.script[s] += list(ops)

    def block(self, active, x, y, n):
        for s in self.script:
            if active[s]:
                self.script[s].append(("mix", n))
                self.x[s].append(x[s])
                self.y[s].append(y[s])

    def check(self, checker):
        for s in self.script:
            if self.x[s]:
                expect = H.run_script_orc(checker, self.fmt, 48000, self.slots, self.script[s], np.concatenate(self.x[s]))
                _assert_exact(expect, np.concatenate(self.y[s]), f"stream {s}")


def _paused_rows_zero(y, active):
    paused = torch.from_numpy(np.flatnonzero(~active)).to(y.device)
    assert not y.index_select(0, paused).view(torch.int32).any().item(), "a paused row is not +0.0f"


def _mix(eng, x, n, layout, host):
    """One block of x ([S][n][C] on the device); returns the output in the same form."""
    if host:
        return torch.from_numpy(eng.mix(x.cpu().numpy())).to(x.device)
    stream = torch.cuda.current_stream().cuda_stream
    if layout == ox.LAYOUT_TILED:
        xt = _to_tiled(x)
        yt = torch.full_like(xt, 1.5)
        eng.mix(xt, yt, frames=n, layout=layout, stream=stream)
        torch.cuda.synchronize()
        return _from_tiled(yt)
    y = torch.full_like(x, 1.5)
    eng.mix(x, y, frames=n, stream=stream)
    torch.cuda.synchronize()
    return y


@pytest.mark.parametrize("layout,host", [(ox.LAYOUT_STREAM_MAJOR, False), (ox.LAYOUT_TILED, False), (ox.LAYOUT_STREAM_MAJOR, True)],
                         ids=["device_stream_major", "device_tiled", "host"])
def test_auto_placement_quarter_active_runs_one_class_per_tile_launch(checker, layout, host):
    """4096 streams of the cfg4 chain, 113 presets as s mod 113, a random quarter active and 64 streams toggled before
    every block, preset changes on paused streams.  Every block (also one that consumes updates) is one kMultiChainStereo
    launch, paused rows are zero, and sampled streams (paused then resumed, changed while paused) are bit-exact."""
    lib = H.cuda_lib()
    S, blocks = 4096, [1024] * 6 + [333]
    rng = np.random.default_rng(25)
    props = [ox.reverb_preset(g, m, lib=lib) for g, m in ox.reverb_preset_names(lib=lib)]
    preset = [s % len(props) for s in range(S)]
    active = np.zeros(S, dtype=bool)
    active[rng.choice(S, S // 4, replace=False)] = True
    # toggles before block b >= 1: 32 paused streams resume, 32 active ones pause
    toggles = {}
    state = active.copy()
    for b in range(1, len(blocks)):
        on = rng.choice(np.flatnonzero(~state), 32, replace=False)
        off = rng.choice(np.flatnonzero(state), 32, replace=False)
        state[on], state[off] = True, False
        toggles[b] = (on, off)
    # preset changes on paused streams before block 2; half of them resume at block 4
    paused_at_2 = np.flatnonzero(~_active_at(active, toggles, 2))
    changed = [int(s) for s in rng.choice(paused_at_2, 16, replace=False)]
    toggles[4] = (np.concatenate([toggles[4][0], changed[:8]]), toggles[4][1])
    resumed = [int(s) for s in toggles[1][0][:6]] + [int(s) for s in toggles[3][0][:4]]
    sample = sorted(set(resumed + changed[:6] + [int(s) for s in toggles[2][1][:4]] +
                        [int(s) for s in np.flatnonzero(active)[:4]] + [0, S - 1]))
    ref = _Streams(sample, F.stereo, 4)
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(4096)
    with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng:
        eng.set_placement("auto")
        for i, t in enumerate(CHAIN[:3]):
            eng.set_effect(i, t)
        for s in range(S):
            eng.set_effect(3, T.eax_reverb, props[preset[s]], first_stream=s, n_streams=1)
            ref.op(s, *[("type", i, t) for i, t in enumerate(CHAIN)], ("props", 3, props[preset[s]]), ("apply",))
        eng.set_active(False)
        for s in np.flatnonzero(active):
            eng.set_active(True, int(s), 1)
        for b, n in enumerate(blocks):
            if b in toggles:
                on, off = toggles[b]
                for s in on:
                    eng.set_active(True, int(s), 1)
                for s in off:
                    eng.set_active(False, int(s), 1)
                active[on], active[off] = True, False
            if b == 2:
                for s in changed:
                    preset[s] = (preset[s] + 17) % len(props)
                    eng.set_effect(3, T.eax_reverb, props[preset[s]], first_stream=s, n_streams=1)
                    ref.op(s, ("props", 3, props[preset[s]]), ("apply",))
            x = torch.rand(S, n, 2, device=dev, generator=gen) - 0.5
            before = eng.launch_count
            y = _mix(eng, x, n, layout, host)
            # (also the blocks that consume updates: the class table carries each class's pending bits)
            assert eng.launch_count - before == 1 and eng.last_kernel == "kMultiChainStereo", (b, eng.launch_count - before, eng.last_kernel)
            _paused_rows_zero(y, active)
            rows = torch.tensor(sample, device=dev)
            ref.block(dict(zip(sample, active[sample])), dict(zip(sample, x[rows].cpu().numpy())), dict(zip(sample, y[rows].cpu().numpy())), n)
    assert all(0 < len(ref.x[s]) < len(blocks) for s in resumed) and all(ref.x[s] for s in changed[:6])
    ref.check(checker)


def _active_at(active, toggles, block):
    state = active.copy()
    for b in range(1, block + 1):
        on, off = toggles[b]
        state[on], state[off] = True, False
    return state


def test_caller_placement_whole_paused_tiles_run_like_a_smaller_engine(checker):
    """cfg2 chain on 4096 streams with 3 of every 4 tiles paused: from the third block on the engine launches what a
    1024-stream engine launches, with the same output bits.  Then single lanes inside active tiles pause as well (the
    masked path) and sampled streams stay bit-exact against the checker."""
    lib = H.cuda_lib()
    S, small_S = 4096, 1024
    tiles = np.arange(S) // 32
    active = tiles % 4 == 1
    lanes_of_small = np.flatnonzero(active)
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(2)
    masked = [int(lanes_of_small[i]) for i in (3, 40, 41, 500, 1023)]
    sample = sorted(set(masked + [int(lanes_of_small[i]) for i in (0, 31, 42, 700)] + [0, 64]))
    ref = _Streams(sample, F.stereo, 4)
    with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng, ox.Engine(small_S, F.stereo, 48000, 4, lib=lib) as small:
        for e in (eng, small):
            for i, t in enumerate(CHAIN):
                e.set_effect(i, t)
        for s in sample:
            ref.op(s, *[("type", i, t) for i, t in enumerate(CHAIN)], ("apply",))
        for t in range(S // 32):
            if t % 4 != 1:
                eng.set_active(False, t * 32, 32)
        for b in range(6):
            if b == 4:
                for s in masked:
                    eng.set_active(False, s, 1)
                    small.set_active(False, int(np.searchsorted(lanes_of_small, s)), 1)
                active[masked] = False
            x = torch.rand(S, 1024, 2, device=dev, generator=gen) - 0.5
            y = _mix(eng, x, 1024, ox.LAYOUT_STREAM_MAJOR, False)
            y_small = _mix(small, x[torch.from_numpy(lanes_of_small).to(dev)].contiguous(), 1024, ox.LAYOUT_STREAM_MAJOR, False)
            if 2 <= b < 4:
                assert eng.last_kernel == small.last_kernel, (b, eng.last_kernel, small.last_kernel)
            _assert_exact(y_small.cpu().numpy(), y[torch.from_numpy(lanes_of_small).to(dev)].cpu().numpy(), f"block {b}")
            _paused_rows_zero(y, active)
            rows = torch.tensor(sample, device=dev)
            ref.block(dict(zip(sample, active[sample])), dict(zip(sample, x[rows].cpu().numpy())), dict(zip(sample, y[rows].cpu().numpy())), 1024)
    ref.check(checker)


def test_span_kernel_runs_with_half_the_tiles_paused(checker):
    """cfg1 (1024 mono EAX reverb streams) with every other tile paused still runs a span kernel and is bit-exact."""
    lib = H.cuda_lib()
    S = 1024
    active = (np.arange(S) // 32) % 2 == 0
    sample = [0, 31, 64, 100, 515, 990, 32, 1023]
    ref = _Streams(sample, F.mono, 1)
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(1)
    with ox.Engine(S, F.mono, 48000, 1, lib=lib) as eng:
        eng.set_effect(0, T.eax_reverb)
        for s in sample:
            ref.op(s, ("type", 0, T.eax_reverb), ("apply",))
        for t in range(1, S // 32, 2):
            eng.set_active(False, t * 32, 32)
        kernels = []
        for b in range(4):
            x = torch.rand(S, 1024, 1, device=dev, generator=gen) - 0.5
            y = _mix(eng, x, 1024, ox.LAYOUT_STREAM_MAJOR, False)
            kernels.append(eng.last_kernel)
            _paused_rows_zero(y, active)
            rows = torch.tensor(sample, device=dev)
            ref.block(dict(zip(sample, active[sample])), dict(zip(sample, x[rows].cpu().numpy())), dict(zip(sample, y[rows].cpu().numpy())), 1024)
    assert kernels[-1].startswith("kSpan"), kernels
    ref.check(checker)


def test_reset_streams_on_the_duo_kernel(checker):
    """16 384 streams of the chain on the duo kernel; single streams and a range across a tile boundary reset after the
    second block.  Each equals its old checker Api up to the reset and a fresh one after it."""
    lib = H.cuda_lib()
    S = 16384
    reset_single, reset_range = [5, 7000], list(range(8190, 8200))
    sample = reset_single + reset_range[:3] + reset_range[-2:] + [0, 8189, S - 1]
    old = _Streams(sample, F.stereo, 4)
    new = _Streams(reset_single + reset_range, F.stereo, 4)
    for s in sample:
        old.op(s, *[("type", i, t) for i, t in enumerate(CHAIN)], ("apply",))
    for s in new.script:
        new.op(s, *[("type", i, t) for i, t in enumerate(CHAIN)], ("apply",))
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(16)
    rows = sorted(set(sample) | set(new.script))
    with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng:
        for i, t in enumerate(CHAIN):
            eng.set_effect(i, t)
        for b in range(5):
            if b == 2:
                for s in reset_single:
                    eng.reset(s, 1)
                eng.reset(reset_range[0], len(reset_range))
            x = torch.rand(S, 1024, 2, device=dev, generator=gen) - 0.5
            y = _mix(eng, x, 1024, ox.LAYOUT_STREAM_MAJOR, False)
            if b == 4:
                assert eng.last_kernel.startswith("kDuo"), eng.last_kernel
            idx = torch.tensor(rows, device=dev)
            xs, ys = dict(zip(rows, x[idx].cpu().numpy())), dict(zip(rows, y[idx].cpu().numpy()))
            # up to the reset every stream is its old Api; after it the reset streams are fresh ones
            old.block({s: b < 2 or s not in new.script for s in sample}, xs, ys, 1024)
            if b >= 2:
                new.block({s: True for s in new.script}, xs, ys, 1024)
    old.check(checker)
    new.check(checker)


def test_mix_bus_sums_the_mixed_streams_only():
    """mix_bus with paused streams (both placements): the bus is bit-identical to reduce_bus of the same output, whose
    paused rows are zero."""
    lib = H.cuda_lib()
    S = 3000
    rng = np.random.default_rng(3)
    active = rng.random(S) >= 0.3
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    for placement in ("caller", "auto"):
        with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng:
            eng.set_placement(placement)
            for i, t in enumerate(CHAIN):
                eng.set_effect(i, t)
            for s in np.flatnonzero(~active):
                eng.set_active(False, int(s), 1)
            for b in range(2):
                x = torch.rand(S, 1024, 2, device=dev) - 0.5
                y = torch.full_like(x, 1.5)
                bus = torch.empty(1024, 2, device=dev)
                bus2 = torch.empty_like(bus)
                eng.mix_bus(x, y, 1024, bus, stream=stream)
                eng.reduce_bus(1024, y, bus2, stream=stream)
                torch.cuda.synchronize()
                _paused_rows_zero(y, active)
                assert torch.equal(bus.view(torch.int32), bus2.view(torch.int32)), (placement, b)

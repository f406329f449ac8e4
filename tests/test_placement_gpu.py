"""Stream placement inside the engine (OALSFX_PLACEMENT_AUTO) on the GPU: voices with arbitrary presets in the caller's
order run on the class-per-tile launch, stay there when presets are re-assigned mid-run, and every caller stream is
bit-exact against the CPU checker and against an unplaced engine."""
import numpy as np
import pytest

import harness as H
import oalsfxpp_b200 as ox
from oalsfxpp_b200 import ChannelFormat as F, EffectType as T

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _lib():
    return H.cuda_lib()


def _assert_match(expect, got, exact, what=""):
    assert expect.shape == got.shape
    if exact:
        e32 = np.ascontiguousarray(expect, dtype=np.float32).view(np.uint32)
        g32 = np.ascontiguousarray(got, dtype=np.float32).view(np.uint32)
        differ = (e32 != g32) & ~(np.isnan(expect) & np.isnan(got))
        if differ.any():
            bad = np.argwhere(differ)
            raise AssertionError((what, "first mismatch at", tuple(bad[0]), "count", len(bad), "max abs diff", H.max_abs_diff(expect, got)))
    else:
        assert H.max_abs_diff(expect, got) <= TOL, (what, H.max_abs_diff(expect, got))


def _to_tiled(x):
    S, frames, C = x.shape
    T_ = (S + 31) // 32
    t = np.zeros((T_ * 32, frames, C), dtype=np.float32)
    t[:S] = x
    return np.ascontiguousarray(t.reshape(T_, 32, frames, C).transpose(0, 2, 3, 1))


def _from_tiled(t, S):
    T_, frames, C, _ = t.shape
    return t.transpose(0, 3, 1, 2).reshape(T_ * 32, frames, C)[:S]


CHAIN = [T.equalizer, T.chorus, T.echo]
N_USER, N_PRESETS = 700, 23
LABELS = np.array([(s * 7 + s // 50) % N_PRESETS for s in range(N_USER)], dtype=np.int32)


def _mix(eng, x, layout):
    if layout == ox.LAYOUT_TILED:
        return _from_tiled(eng.mix(_to_tiled(x), layout=layout), x.shape[0])
    return eng.mix(np.ascontiguousarray(x))


@pytest.mark.parametrize("layout", [ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED], ids=["stream_major", "tiled"])
def test_auto_placement_runs_arbitrary_presets_in_caller_order_on_one_launch(checker, layout):
    """700 voices, 23 reverb presets in no particular order, buffers in the caller's order: every block is ONE
    kMultiChainStereo launch, and sampled caller streams are bit-exact."""
    lib = _lib()
    names = ox.reverb_preset_names(lib=lib)
    props = {p: ox.reverb_preset(*names[(p * 5) % len(names)], lib=lib) for p in range(N_PRESETS)}
    blocks = [1024, 333]
    x = np.stack([H.noise(7000 + s, 2, sum(blocks)) for s in range(N_USER)])
    y = np.empty_like(x)
    with ox.Engine(N_USER, F.stereo, 48000, 4, lib=lib) as eng:
        eng.set_placement("auto")
        for i, t in enumerate(CHAIN):
            eng.set_effect(i, t)
        for s in range(N_USER):
            eng.set_effect(3, T.eax_reverb, props[int(LABELS[s])], first_stream=s, n_streams=1)
        at = 0
        for n in blocks:
            before = eng.launch_count
            y[:, at:at + n] = _mix(eng, x[:, at:at + n], layout)
            assert eng.launch_count - before == 1 and eng.last_kernel == "kMultiChainStereo", (eng.launch_count - before, eng.last_kernel)
            at += n
        lanes, count = eng.lanes()
        assert count % 32 == 0 and len(set(lanes.tolist())) == N_USER
    for s in (0, 1, 49, 50, 333, N_USER - 1):
        script = H.simple_script([(t, None) for t in CHAIN] + [(T.eax_reverb, props[int(LABELS[s])])], blocks)
        expect = H.run_script_orc(checker, F.stereo, 48000, 4, script, x[s])
        _assert_match(expect, y[s], True, f"caller stream {s}")


def test_auto_placement_keeps_one_launch_after_mid_run_reassignment(checker):
    """After block 2, 37 scattered voices move to other presets or new properties and some of them change chorus ->
    flanger.  From the block after the update on no table-mode kernel runs and every block is one launch; changed and
    unchanged voices are bit-exact, and their integer state equals an unplaced engine's."""
    lib = _lib()
    names = ox.reverb_preset_names(lib=lib)
    props = {p: ox.reverb_preset(*names[(p * 5) % len(names)], lib=lib) for p in range(N_PRESETS)}
    rng = np.random.default_rng(37)
    moved = sorted(int(s) for s in rng.choice(N_USER, 37, replace=False))
    new_props = {}
    for i, s in enumerate(moved):
        if i % 3 == 2:   # new properties nobody had
            new_props[s] = ox.default_props(T.eax_reverb, lib=lib, decay_time_=0.7 + 0.05 * i, gain_=0.2)
        else:
            new_props[s] = props[(int(LABELS[s]) + 1 + i) % N_PRESETS]
    flanger = set(moved[::4])
    blocks = [1024, 1024, 1024, 1024, 512]
    x = np.stack([H.noise(8000 + s, 2, sum(blocks)) for s in range(N_USER)])
    y = np.empty_like(x)
    ref_state = {}
    sample = sorted({0, 1, 50, 333, N_USER - 1, moved[0], moved[1], moved[2], moved[4], moved[5]})
    with ox.Engine(N_USER, F.stereo, 48000, 4, lib=lib) as eng, ox.Engine(N_USER, F.stereo, 48000, 4, lib=lib) as ref:
        eng.set_placement("auto")
        for e in (eng, ref):
            for i, t in enumerate(CHAIN):
                e.set_effect(i, t)
            for s in range(N_USER):
                e.set_effect(3, T.eax_reverb, props[int(LABELS[s])], first_stream=s, n_streams=1)
        at = 0
        for b, n in enumerate(blocks):
            if b == 2:
                for e in (eng, ref):
                    for s in moved:
                        e.set_effect(3, T.eax_reverb, new_props[s], first_stream=s, n_streams=1)
                        if s in flanger:
                            e.set_effect(1, T.flanger, first_stream=s, n_streams=1)
            before = eng.launch_count
            xb = np.ascontiguousarray(x[:, at:at + n])
            y[:, at:at + n] = eng.mix(xb)
            ref.mix(xb)
            if b >= 3:
                assert eng.launch_count - before == 1 and not eng.last_kernel.startswith("kTab"), (b, eng.launch_count - before, eng.last_kernel)
            at += n
        for s in sample:
            for slot in range(4):
                assert eng.debug_state(s, slot) == ref.debug_state(s, slot), (s, slot)
    for s in sample:
        script = [("type", i, t) for i, t in enumerate(CHAIN)] + [("type", 3, T.eax_reverb), ("props", 3, props[int(LABELS[s])]), ("apply",)]
        for b, n in enumerate(blocks):
            if b == 2 and s in new_props:
                script += [("props", 3, new_props[s])]
                if s in flanger:
                    script += [("type", 1, T.flanger)]
                script += [("apply",)]
            script.append(("mix", n))
        expect = H.run_script_orc(checker, F.stereo, 48000, 4, script, x[s])
        _assert_match(expect, y[s], True, f"caller stream {s}")


def _two_signatures(lib, s, phase):
    default = lambda t, **kw: ox.default_props(t, lib=lib, **kw)
    if s % 5 == 4:
        return [(T.flanger, default(T.flanger, rate_=0.1 + 0.01 * s)), (T.ring_modulator, default(T.ring_modulator, frequency_=300.0 + 7 * s)),
                (T.distortion, default(T.distortion, edge_=0.1 + 0.005 * (s % 100))), (T.compressor, None)]
    return [(T.equalizer, default(T.equalizer, mid1_gain_=0.5 + 0.01 * s + 0.2 * phase)), (T.chorus, default(T.chorus, depth_=0.05 + 0.001 * s)),
            (T.echo, default(T.echo, delay_=0.02 + 0.001 * s, feedback_=0.3)),
            (T.eax_reverb if s % 2 else T.reverb, default(T.eax_reverb if s % 2 else T.reverb, gain_=0.1 + 0.002 * s,
                                                           decay_time_=0.5 + 0.01 * s + 0.3 * phase, reflections_delay_=0.001 * (s % 20)))]


def test_auto_placement_gives_each_slot_signature_one_launch(checker):
    """The configuration of the table-mode test (1000 voices, each its own parameters, two slot signatures, a change
    of parameters after the first block), without its send filters: placed, a steady block takes at most one launch
    per signature.  Bit-exact, the ring-modulator voices within 1e-5 (the device sinf)."""
    lib = _lib()
    S, block, nblocks = 1000, 512, 3
    x = np.stack([H.noise(500 + s, 2, block * nblocks) for s in range(S)])
    y = np.empty_like(x)
    with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng:
        eng.set_placement("auto")
        for s in range(S):
            for slot, (t, p) in enumerate(_two_signatures(lib, s, 0)):
                eng.set_effect(slot, t, p, first_stream=s, n_streams=1)
        for b in range(nblocks):
            if b == 1:
                for s in range(S):
                    for slot, (t, p) in enumerate(_two_signatures(lib, s, 1)):
                        eng.set_effect(slot, t, p, first_stream=s, n_streams=1)
            before = eng.launch_count
            y[:, b * block:(b + 1) * block] = eng.mix(np.ascontiguousarray(x[:, b * block:(b + 1) * block]))
            if b == nblocks - 1:
                assert eng.launch_count - before <= 2, eng.launch_count - before
    for s in (0, 1, 4, 7, 31, 32, 333, 504, 998, 999):
        script = []
        for slot, (t, p) in enumerate(_two_signatures(lib, s, 0)):
            script += [("type", slot, t)] + ([("props", slot, p)] if p is not None else [])
        script += [("apply",), ("mix", block)]
        for slot, (t, p) in enumerate(_two_signatures(lib, s, 1)):
            script += [("type", slot, t)] + ([("props", slot, p)] if p is not None else [])
        script += [("apply",)] + [("mix", block)] * (nblocks - 1)
        expect = H.run_script_orc(checker, F.stereo, 48000, 4, script, x[s])
        _assert_match(expect, y[s], s % 5 != 4, f"stream {s}")


def test_auto_to_caller_placement_continues_as_a_never_placed_engine():
    """Device buffers (torch), both layouts: after AUTO -> CALLER the lanes are the identity again, the output continues
    bit for bit as a never-placed engine's, and the same kernel serves the block."""
    torch = pytest.importorskip("torch")
    lib = _lib()
    names = ox.reverb_preset_names(lib=lib)
    S, frames = 200, 512
    labels = [(s * 3) % 11 for s in range(S)]
    props = {p: ox.reverb_preset(*names[p * 3], lib=lib) for p in range(11)}
    for layout in (ox.LAYOUT_STREAM_MAJOR, ox.LAYOUT_TILED):
        with ox.Engine(S, F.stereo, 48000, 4, lib=lib) as eng, ox.Engine(S, F.stereo, 48000, 4, lib=lib) as ref:
            eng.set_placement("auto")
            for e in (eng, ref):
                for i, t in enumerate(CHAIN):
                    e.set_effect(i, t)
                for s in range(S):
                    e.set_effect(3, T.eax_reverb, props[labels[s]], first_stream=s, n_streams=1)
            for b in range(4):
                if b == 2:
                    eng.set_placement("caller")
                    lanes, count = eng.lanes()
                    assert lanes.tolist() == list(range(S)) and count == (S + 31) // 32 * 32
                x = np.stack([H.noise(100 * b + s, 2, frames) for s in range(S)])
                if layout == ox.LAYOUT_TILED:
                    x = _to_tiled(x)
                src = torch.from_numpy(x).cuda()
                out = [torch.zeros_like(src) for _ in range(2)]
                eng.mix(src, out[0], frames=frames, layout=layout)
                ref.mix(src, out[1], frames=frames, layout=layout)
                torch.cuda.synchronize()
                a, r = out[0].cpu().numpy(), out[1].cpu().numpy()
                if layout == ox.LAYOUT_TILED:
                    a, r = _from_tiled(a, S), _from_tiled(r, S)
                _assert_match(r, a, True, f"layout {layout} block {b}")
                if b >= 2:
                    assert eng.last_kernel == ref.last_kernel, (eng.last_kernel, ref.last_kernel)


def test_placed_snapshot_equals_unplaced_and_restores_across_modes():
    lib = _lib()
    names = ox.reverb_preset_names(lib=lib)
    S, frames = 96, 700
    props = {p: ox.reverb_preset(*names[p * 2], lib=lib) for p in range(7)}

    def configure(e, labels):
        for i, t in enumerate(CHAIN):
            e.set_effect(i, t)
        for s in range(S):
            e.set_effect(3, T.eax_reverb, props[labels[s]], first_stream=s, n_streams=1)

    labels = [(s * 5) % 7 for s in range(S)]
    engines = [ox.Engine(S, F.stereo, 48000, 4, lib=lib) for _ in range(4)]
    try:
        placed, plain, plain2, placed2 = engines
        placed.set_placement("auto")
        placed2.set_placement("auto")
        for e in engines:
            configure(e, labels)
        for b in range(3):
            x = np.stack([H.noise(40 * b + s, 2, frames) for s in range(S)])
            if b == 1:
                for e in (placed, plain):
                    e.set_effect(3, T.eax_reverb, props[6], first_stream=10, n_streams=3)
                    e.set_effect(1, T.flanger, first_stream=50, n_streams=1)
            ya, yb = placed.mix(x), plain.mix(x)
            _assert_match(yb, ya, True, f"block {b}")
        assert placed.lane_of_stream.tolist() != list(range(S))
        snap_placed, snap_plain = placed.snapshot(), plain.snapshot()
        assert np.array_equal(snap_placed, snap_plain)
        for e in (plain2, placed2):   # same configuration as the snapshotted pair
            e.set_effect(3, T.eax_reverb, props[6], first_stream=10, n_streams=3)
            e.set_effect(1, T.flanger, first_stream=50, n_streams=1)
        plain2.restore(snap_placed)
        placed2.restore(snap_plain)
        for b in range(3, 5):
            x = np.stack([H.noise(40 * b + s, 2, frames) for s in range(S)])
            outs = [e.mix(x) for e in engines]
            for i in (0, 2, 3):
                _assert_match(outs[1], outs[i], True, f"engine {i} block {b}")
    finally:
        for e in engines:
            e.close()

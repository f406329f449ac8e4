"""Pins the CPU checkers (test infrastructure under oracle/).

  * the hand-written restatement (oracle/oalsfx_oracle.cpp) == the committed golden vectors that were
    produced by the compiled reference (tests/golden/make_golden.py) -- runs everywhere;
  * the restatement == the compiled reference, bit for bit, over the whole case matrix, and the
    compiled reference == the golden vectors -- runs wherever oracle/_ref exists (build container and,
    because the .so travels, the GPU box).
"""
import hashlib
import os

import numpy as np
import pytest

import cases
import harness as H

GOLDEN = np.load(os.path.join(H.ROOT, "tests", "golden", "golden.npz"))
QUICK = list(cases.all_cases(H.emu_lib(), quick=True))


def _sha(y):
    return np.frombuffer(hashlib.sha256(y.tobytes()).digest(), dtype=np.uint8)


@pytest.mark.parametrize("case", QUICK, ids=[c[0] for c in QUICK])
def test_restatement_matches_golden(case):
    name, fmt, rate, effect_count, script, x = case
    y = H.run_script_orc(H.oracle_lib(), fmt, rate, effect_count, script, x)
    if "full/" + name in GOLDEN:
        want = GOLDEN["full/" + name]
        assert y.shape == want.shape
        assert np.array_equal(np.isnan(y), np.isnan(want))
        assert H.max_abs_diff(np.nan_to_num(y), np.nan_to_num(want)) <= 1e-6
    assert np.array_equal(_sha(y), GOLDEN["sha256/" + name]), "output differs from the reference-generated golden hash"


def test_reference_matches_golden(ref):
    """The golden hashes and the POD sizes test_abi.py pins (108 / 112 bytes) are what the compiled reference gives."""
    for name, fmt, rate, effect_count, script, x in QUICK:
        y = H.run_script_orc(ref, fmt, rate, effect_count, script, x)
        assert np.array_equal(_sha(y), GOLDEN["sha256/" + name]), name
    assert ref.orc_sizeof_effect_props() == 108 and ref.orc_sizeof_effect() == 112


def test_restatement_matches_reference_on_full_matrix(ref):
    orc = H.oracle_lib()
    for name, fmt, rate, effect_count, script, x in cases.all_cases(H.emu_lib(), quick=False):
        a = H.run_script_orc(ref, fmt, rate, effect_count, script, x)
        b = H.run_script_orc(orc, fmt, rate, effect_count, script, x)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name


def test_restatement_ten_seconds_chain(ref):
    """10 s of the 4-slot stereo chain in 1024-frame blocks: restatement == reference."""
    from oalsfxpp_b200.props import ChannelFormat as F, EffectType as T
    total = 480000
    x = H.noise(77, 2, total)
    script = H.simple_script([(T.equalizer, None), (T.chorus, None), (T.echo, None), (T.eax_reverb, None)],
                             H.blocks_of(total, 1024))
    a = H.run_script_orc(ref, F.stereo, 48000, 4, script, x)
    b = H.run_script_orc(H.oracle_lib(), F.stereo, 48000, 4, script, x)
    assert np.array_equal(a, b)


def test_noise_generators_agree():
    """The hash noise is identical in numpy (tests), the C shim the reference is wrapped with (oracle/ref_shim.cpp,
    here compiled against include/oalsfxpp.h) and the restatement."""
    want = H.noise(5, 2, 1000, first_frame=123)
    for lib in (H.api_shim("emu"), H.oracle_lib()):
        got = np.zeros((1000, 2), np.float32)
        lib.orc_noise(H.SEED, 5, 2, 123, 1000, got.ctypes.data)
        assert np.array_equal(want, got)
    assert want.min() >= -0.5 and want.max() < 0.5

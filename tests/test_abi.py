"""The C-ABI library loads and exports every symbol include/oalsfx_engine.h declares (no compute)."""
import ctypes
import os
import re

import harness as H
from oalsfxpp_b200 import engine as E


def _declared_symbols():
    text = open(os.path.join(H.ROOT, "include", "oalsfx_engine.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(oalsfx_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_match_binding_list():
    assert _declared_symbols() == sorted(E.EXPORTED_SYMBOLS)


def test_product_library_exports_every_symbol():
    path = E.library_path()
    assert os.path.exists(path), "build the CUDA library first (__graft_entry__.build())"
    lib = ctypes.CDLL(path)
    for name in _declared_symbols():
        assert hasattr(lib, name), name
    info = ctypes.c_char_p(ctypes.cast(lib.oalsfx_build_info, ctypes.CFUNCTYPE(ctypes.c_char_p))()).value
    assert b"sm_100a" in info and b"cuda" in info


def test_product_library_also_exports_the_cpp_api():
    """The drop-in class: mangled oalsfxpp::Api members are exported (reference: oalsfxpp.h:760-922)."""
    import subprocess
    out = subprocess.run(["nm", "-DC", E.library_path()], check=True, capture_output=True, text=True).stdout
    for member in ("oalsfxpp::Api::initialize(", "oalsfxpp::Api::mix(int, float const*, float*)",
                   "oalsfxpp::Api::apply_changes()", "oalsfxpp::Api::set_effect_props(",
                   "oalsfxpp::Api::set_send_props(", "oalsfxpp::Effect::set_type_and_defaults(",
                   "oalsfxpp::ReverbPresets::Default::generic", "oalsfxpp::EffectProps::Reverb::normalize()"):
        assert member in out, member


def test_no_cpu_fallback_without_a_gpu():
    """Creating an engine must fail loudly when no CUDA device is usable."""
    import pytest
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    import oalsfxpp_b200 as ox
    with pytest.raises(ox.OalsfxError) as err:
        ox.Engine(4, ox.ChannelFormat.stereo, 48000, 1)
    assert "no CPU fallback" in str(err.value)


def test_pod_layout_matches_reference():
    """sizeof(EffectProps)=108, sizeof(Effect)=112 as measured on the reference (SURVEY.md section 2; checked against the
    compiled reference by test_oracle.py::test_reference_matches_golden)."""
    assert ctypes.sizeof(E.EffectProps) == 108
    shim = H.api_shim("emu")
    assert shim.orc_sizeof_effect_props() == 108 and shim.orc_sizeof_effect() == 112


def test_plan_placement_is_a_pure_host_function():
    """oalsfx_plan_placement needs no engine and no device: callable on the PRODUCT library without a GPU.  Classes in
    order of first appearance, each range a multiple of 32, caller order kept inside a class; bad arguments are refused."""
    import numpy as np
    import oalsfxpp_b200 as ox
    lib = E.bind(ctypes.CDLL(E.library_path()))
    labels = np.array([7, 7, 3, 7, 3, 9] + [3] * 40, dtype=np.int32)
    index, total, classes = ox.plan_placement(labels, lib=lib)
    assert classes == [(7, 0, 32), (3, 32, 64), (9, 96, 32)] and total == 128
    assert index[:6].tolist() == [0, 1, 32, 2, 33, 96] and index[6:].tolist() == list(range(34, 74))
    one, total1, classes1 = ox.plan_placement(np.zeros(65, dtype=np.int32), lib=lib)
    assert total1 == 96 and classes1 == [(0, 0, 96)] and one.tolist() == list(range(65))
    out = (ctypes.c_int32 * 4)()
    assert lib.oalsfx_plan_placement(None, 4, out, None, 0, None) < 0
    assert lib.oalsfx_plan_placement(out, 0, out, None, 0, None) < 0
    assert lib.oalsfx_plan_placement(out, 4, out, None, 3, None) < 0   # a capacity without a buffer

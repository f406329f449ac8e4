"""oalsfxpp_b200 -- Python host-side binding of the B200-native batched effects engine.

The product is the shared library ``liboalsfx_b200.so`` (CUDA kernels for sm_100a + the C ABI of
``include/oalsfx_engine.h`` + the drop-in C++ class ``oalsfxpp::Api`` of ``include/oalsfxpp.h``).
This package only binds the C ABI with ctypes for tests and benchmarks; it contains no signal
processing of its own and there is no CPU fallback: importing works anywhere, but creating an
:class:`Engine` raises unless the CUDA library is built and a GPU is present.
"""
from .props import (ChannelFormat, EffectType, EffectProps, channel_count, default_props,
                    normalize_props, reverb_preset, reverb_preset_names)
from .engine import (Engine, OalsfxError, LAYOUT_STREAM_MAJOR, LAYOUT_TILED, BUS_NONE, MAX_ROUTES, SPACE_HOST,
                     SPACE_DEVICE, library_path, load_library, build_info, plan_placement)

__all__ = [
    "ChannelFormat", "EffectType", "EffectProps", "channel_count", "default_props",
    "normalize_props", "reverb_preset", "reverb_preset_names", "Engine", "OalsfxError",
    "LAYOUT_STREAM_MAJOR", "LAYOUT_TILED", "BUS_NONE", "MAX_ROUTES", "SPACE_HOST", "SPACE_DEVICE", "library_path",
    "load_library", "build_info", "plan_placement",
]

"""ctypes binding of include/oalsfx_engine.h.

:class:`Engine` mirrors, for a batch of streams, what one ``oalsfxpp::Api`` instance does for one
(reference: src/oalsfxpp.h:760-922): ``set_effect`` = ``set_effect_type``/``set_effect_props`` +
``apply_changes`` for a stream range, ``set_sends`` = ``set_send_props`` + ``apply_changes``,
``mix`` = ``Api::mix`` for all streams at once.  Error behaviour follows the C ABI: a non-zero
code raises :class:`OalsfxError` with the library's message.
"""
import ctypes as C
import os

import numpy as np

from .props import EffectProps, EffectType, channel_count

LAYOUT_STREAM_MAJOR = 0
LAYOUT_TILED = 1
BUS_NONE = -1
MAX_ROUTES = 4
SPACE_HOST = 0
SPACE_DEVICE = 1


class OalsfxError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"oalsfx error {code}: {message}")
        self.code = code
        self.message = message


class _Desc(C.Structure):
    _fields_ = [("device", C.c_int32), ("num_streams", C.c_int32), ("channel_format", C.c_int32),
                ("sampling_rate", C.c_int32), ("effect_count", C.c_int32)]


def library_path():
    """The in-tree CUDA library.  OALSFX_LIB may name another build of the SAME library (A/B kernel
    tuning builds made by oalsfxpp_b200/csrc/Makefile with different -D flags); it is never a fallback."""
    override = os.environ.get("OALSFX_LIB")
    if override:
        return os.path.abspath(override)
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "liboalsfx_b200.so")


def bind(lib):
    """Declare the prototypes of every symbol include/oalsfx_engine.h exports."""
    vp, i32, f32p = C.c_void_p, C.c_int, C.POINTER(C.c_float)
    lib.oalsfx_engine_create.argtypes = [C.POINTER(_Desc), C.POINTER(vp)]
    lib.oalsfx_engine_create.restype = i32
    lib.oalsfx_engine_destroy.argtypes = [vp]
    lib.oalsfx_engine_destroy.restype = None
    lib.oalsfx_engine_set_effect.argtypes = [vp, i32, i32, i32, i32, vp, C.c_size_t]
    lib.oalsfx_engine_set_effect.restype = i32
    lib.oalsfx_engine_set_sends.argtypes = [vp, i32, i32, f32p, f32p]
    lib.oalsfx_engine_set_sends.restype = i32
    lib.oalsfx_engine_set_active.argtypes = [vp, i32, i32, i32]
    lib.oalsfx_engine_set_active.restype = i32
    lib.oalsfx_engine_reset_streams.argtypes = [vp, i32, i32]
    lib.oalsfx_engine_reset_streams.restype = i32
    lib.oalsfx_engine_mix.argtypes = [vp, i32, vp, vp, i32, i32, vp]
    lib.oalsfx_engine_mix.restype = i32
    lib.oalsfx_engine_pin_host.argtypes = [vp, vp, C.c_size_t]
    lib.oalsfx_engine_pin_host.restype = i32
    lib.oalsfx_engine_unpin_host.argtypes = [vp, vp]
    lib.oalsfx_engine_unpin_host.restype = i32
    lib.oalsfx_engine_mix_bus.argtypes = [vp, i32, vp, vp, i32, vp, vp]
    lib.oalsfx_engine_mix_bus.restype = i32
    lib.oalsfx_engine_reduce_bus.argtypes = [vp, i32, vp, i32, vp, vp]
    lib.oalsfx_engine_reduce_bus.restype = i32
    lib.oalsfx_engine_route_streams.argtypes = [vp, i32, i32, vp]
    lib.oalsfx_engine_route_streams.restype = i32
    lib.oalsfx_engine_set_routes.argtypes = [vp, i32, i32, i32, vp, vp, i32]
    lib.oalsfx_engine_set_routes.restype = i32
    lib.oalsfx_engine_set_bus_format.argtypes = [vp, i32]
    lib.oalsfx_engine_set_bus_format.restype = i32
    lib.oalsfx_engine_set_route_pans.argtypes = [vp, i32, i32, i32, vp, vp, i32]
    lib.oalsfx_engine_set_route_pans.restype = i32
    lib.oalsfx_engine_reduce_buses.argtypes = [vp, i32, vp, i32, i32, vp, vp]
    lib.oalsfx_engine_reduce_buses.restype = i32
    lib.oalsfx_engine_mix_buses.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp]
    lib.oalsfx_engine_mix_buses.restype = i32
    lib.oalsfx_engine_debug_state.argtypes = [vp, i32, i32, C.POINTER(C.c_int32)]
    lib.oalsfx_engine_debug_state.restype = i32
    lib.oalsfx_engine_launch_count.argtypes = [vp]
    lib.oalsfx_engine_launch_count.restype = C.c_longlong
    lib.oalsfx_engine_last_kernel.argtypes = [vp]
    lib.oalsfx_engine_last_kernel.restype = C.c_char_p
    lib.oalsfx_engine_device_bytes.argtypes = [vp]
    lib.oalsfx_engine_device_bytes.restype = C.c_longlong
    lib.oalsfx_last_error.argtypes = [vp]
    lib.oalsfx_last_error.restype = C.c_char_p
    lib.oalsfx_build_info.argtypes = []
    lib.oalsfx_build_info.restype = C.c_char_p
    lib.oalsfx_effect_defaults.argtypes = [i32, vp, C.c_size_t]
    lib.oalsfx_effect_defaults.restype = i32
    lib.oalsfx_effect_normalize.argtypes = [i32, vp, C.c_size_t]
    lib.oalsfx_effect_normalize.restype = i32
    lib.oalsfx_reverb_preset.argtypes = [C.c_char_p, C.c_char_p, vp, C.c_size_t]
    lib.oalsfx_reverb_preset.restype = i32
    lib.oalsfx_reverb_preset_name.argtypes = [i32]
    lib.oalsfx_reverb_preset_name.restype = C.c_char_p
    lib.oalsfx_pcm_to_float.argtypes = [vp, vp, i32, vp, C.c_longlong, vp]
    lib.oalsfx_pcm_to_float.restype = i32
    lib.oalsfx_debug_waveshaper.argtypes = [vp, vp, C.c_float, vp, C.c_longlong, vp]
    lib.oalsfx_debug_waveshaper.restype = i32
    lib.oalsfx_plan_placement.argtypes = [vp, i32, vp, vp, i32, vp]
    lib.oalsfx_plan_placement.restype = C.c_longlong
    lib.oalsfx_float_to_s16.argtypes = [vp, vp, vp, i32, C.c_longlong, vp, vp]
    lib.oalsfx_float_to_s16.restype = i32
    lib.oalsfx_engine_snapshot_size.argtypes = [vp]
    lib.oalsfx_engine_snapshot_size.restype = C.c_longlong
    lib.oalsfx_engine_snapshot.argtypes = [vp, vp, C.c_size_t]
    lib.oalsfx_engine_snapshot.restype = i32
    lib.oalsfx_engine_restore.argtypes = [vp, vp, C.c_size_t]
    lib.oalsfx_engine_restore.restype = i32
    lib.oalsfx_engine_set_placement.argtypes = [vp, i32]
    lib.oalsfx_engine_set_placement.restype = i32
    lib.oalsfx_engine_lanes.argtypes = [vp, vp, i32]
    lib.oalsfx_engine_lanes.restype = C.c_longlong
    return lib


EXPORTED_SYMBOLS = (
    "oalsfx_engine_create", "oalsfx_engine_destroy", "oalsfx_engine_set_effect",
    "oalsfx_engine_set_sends", "oalsfx_engine_set_active", "oalsfx_engine_reset_streams", "oalsfx_engine_mix", "oalsfx_engine_mix_bus", "oalsfx_engine_reduce_bus",
    "oalsfx_engine_route_streams", "oalsfx_engine_set_routes", "oalsfx_engine_set_bus_format",
    "oalsfx_engine_set_route_pans", "oalsfx_engine_reduce_buses", "oalsfx_engine_mix_buses",
    "oalsfx_engine_pin_host", "oalsfx_engine_unpin_host",
    "oalsfx_engine_debug_state", "oalsfx_debug_waveshaper", "oalsfx_plan_placement", "oalsfx_engine_launch_count", "oalsfx_engine_last_kernel", "oalsfx_engine_device_bytes",
    "oalsfx_last_error", "oalsfx_build_info", "oalsfx_effect_defaults", "oalsfx_effect_normalize",
    "oalsfx_reverb_preset", "oalsfx_reverb_preset_name", "oalsfx_pcm_to_float", "oalsfx_float_to_s16",
    "oalsfx_engine_snapshot_size", "oalsfx_engine_snapshot", "oalsfx_engine_restore",
    "oalsfx_engine_set_placement", "oalsfx_engine_lanes",
)

_LIB = None


def load_library():
    """Load the CUDA library built in-tree.  Fails loudly when it is missing: there is no fallback."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise OalsfxError(-5, f"{path} is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                                  "the engine has no CPU fallback")
        _LIB = bind(C.CDLL(path))
    return _LIB


def plan_placement(labels, lib=None):
    """oalsfx_plan_placement: an engine stream index per caller stream such that every 32-stream tile holds one class.
    Returns (index array, engine stream count, [(label, first engine index, range length incl. padding), ...])."""
    lib = lib or load_library()
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    index = np.empty(labels.size, dtype=np.int32)
    triples = np.empty((max(1, labels.size), 3), dtype=np.int32)
    n_classes = C.c_int(0)
    total = lib.oalsfx_plan_placement(labels.ctypes.data, int(labels.size), index.ctypes.data, triples.ctypes.data,
                                      int(triples.shape[0]), C.addressof(n_classes))
    if total < 0:
        raise OalsfxError(int(total), "oalsfx_plan_placement: bad arguments")
    return index, int(total), [tuple(int(v) for v in t) for t in triples[:n_classes.value]]


def build_info(lib=None):
    return (lib or load_library()).oalsfx_build_info().decode()


def _ptr(buf):
    """Raw address of a numpy array, a torch tensor or an int."""
    if isinstance(buf, int):
        return buf
    if isinstance(buf, np.ndarray):
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):
        return buf.data_ptr()
    raise TypeError(type(buf))


class Engine:
    """``num_streams`` independent streams, each equivalent to one reference ``Api`` instance."""

    def __init__(self, num_streams, channel_format, sampling_rate, effect_count, device=0, lib=None):
        self.lib = lib if lib is not None else load_library()
        self.num_streams = int(num_streams)
        self.channel_format = int(channel_format)
        self.channels = channel_count(channel_format)
        self.sampling_rate = int(sampling_rate)
        self.effect_count = int(effect_count)
        self.bus_format = self.channel_format
        desc = _Desc(int(device), self.num_streams, self.channel_format, self.sampling_rate, self.effect_count)
        handle = C.c_void_p()
        rc = self.lib.oalsfx_engine_create(C.byref(desc), C.byref(handle))
        if rc != 0:
            raise OalsfxError(rc, self.lib.oalsfx_last_error(None).decode())
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self.lib.oalsfx_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise OalsfxError(rc, self.lib.oalsfx_last_error(self._h).decode())

    @property
    def padded_streams(self):
        return (self.num_streams + 31) // 32 * 32

    def set_effect(self, slot, effect_type, props=None, first_stream=0, n_streams=None):
        """Slot `slot` of the stream range becomes `effect_type` with `props` (defaults if None)."""
        n = self.num_streams - first_stream if n_streams is None else n_streams
        if props is None and int(effect_type) != int(EffectType.null):
            props = EffectProps()
            self.lib.oalsfx_effect_defaults(int(effect_type), C.byref(props), C.sizeof(props))
        if props is None:
            self._check(self.lib.oalsfx_engine_set_effect(self._h, first_stream, n, slot, int(effect_type), None, 0))
        else:
            self._check(self.lib.oalsfx_engine_set_effect(self._h, first_stream, n, slot, int(effect_type),
                                                          C.addressof(props), C.sizeof(props)))

    def set_sends(self, direct=(1.0, 1.0, 1.0), aux=None, first_stream=0, n_streams=None):
        """direct = (gain, gain_hf, gain_lf); aux = one such triple per slot."""
        n = self.num_streams - first_stream if n_streams is None else n_streams
        aux = aux if aux is not None else [(1.0, 1.0, 1.0)] * self.effect_count
        d = (C.c_float * 3)(*direct)
        flat = [v for triple in aux for v in triple]
        a = (C.c_float * len(flat))(*flat)
        self._check(self.lib.oalsfx_engine_set_sends(self._h, first_stream, n, d, a))

    def set_active(self, active, first_stream=0, n_streams=None):
        """Mix (True) or pause (False) the stream range.  A paused stream keeps all of its state, its input is not read and
        its output rows are zeros; it resumes bit for bit where it stopped."""
        n = self.num_streams - first_stream if n_streams is None else n_streams
        self._check(self.lib.oalsfx_engine_set_active(self._h, first_stream, n, 1 if active else 0))

    def reset(self, first_stream=0, n_streams=None):
        """The stream range restarts from silence with its current effects and sends, like a freshly created engine."""
        n = self.num_streams - first_stream if n_streams is None else n_streams
        self._check(self.lib.oalsfx_engine_reset_streams(self._h, first_stream, n))

    def mix(self, src, dst=None, frames=None, layout=LAYOUT_STREAM_MAJOR, space=None, stream=0):
        """Api::mix for every stream.  numpy arrays are host buffers, torch CUDA tensors device buffers."""
        if space is None:
            space = SPACE_HOST if isinstance(src, np.ndarray) else SPACE_DEVICE
        if isinstance(src, np.ndarray):
            src = np.ascontiguousarray(src, dtype=np.float32)
            if frames is None:
                frames = src.size // (self.channels * (self.padded_streams if layout == LAYOUT_TILED else self.num_streams))
            if dst is None:
                dst = np.empty_like(src)
            elif not (isinstance(dst, np.ndarray) and dst.dtype == np.float32 and dst.flags["C_CONTIGUOUS"] and dst.size == src.size):
                raise ValueError("dst must be a C-contiguous float32 array of the same size as src")
        elif frames is None:
            raise ValueError("frames is required for raw / device buffers")
        self._check(self.lib.oalsfx_engine_mix(self._h, int(frames), _ptr(src), _ptr(dst), layout, space,
                                               C.c_void_p(stream)))
        return dst

    def pin_host(self, array):
        """Page-lock a numpy buffer in place (see oalsfx_engine_pin_host); keep it alive until unpin_host / close."""
        self._check(self.lib.oalsfx_engine_pin_host(self._h, array.ctypes.data, array.nbytes))

    def unpin_host(self, array):
        self._check(self.lib.oalsfx_engine_unpin_host(self._h, array.ctypes.data))

    def mix_bus(self, src, dst, frames, bus, layout=LAYOUT_STREAM_MAJOR, stream=0):
        """mix() on device buffers that also fills `bus` ([frames][channels], device) with the sum of the output over all
        streams -- an epilogue of the fused kernel where that serves the whole engine."""
        self._check(self.lib.oalsfx_engine_mix_bus(self._h, int(frames), _ptr(src), _ptr(dst), layout, _ptr(bus),
                                                   C.c_void_p(stream)))
        return bus

    def reduce_bus(self, frames, dst, bus, layout=LAYOUT_STREAM_MAJOR, stream=0):
        self._check(self.lib.oalsfx_engine_reduce_bus(self._h, int(frames), _ptr(dst), layout, _ptr(bus),
                                                      C.c_void_p(stream)))
        return bus

    def route(self, bus, first_stream=0):
        """Route streams first_stream, first_stream + 1, ... to the buses in `bus` (ints; BUS_NONE = -1: no bus)."""
        bus = np.ascontiguousarray(bus, dtype=np.int32).ravel()
        self._check(self.lib.oalsfx_engine_route_streams(self._h, int(first_stream), int(bus.size), bus.ctypes.data))

    def set_routes(self, bus, gain=None, first_stream=0, ramp_frames=0):
        """Routes of streams first_stream, first_stream + 1, ...: bus[i] (up to MAX_ROUTES bus indices, BUS_NONE for none)
        with gains gain[i] (default 1.0), each gain ramped from the route's current one over ramp_frames frames (a new
        route from 0).  `bus` and `gain` are [n][R] arrays; a 1-D array means one route per stream."""
        bus = np.asarray(bus, dtype=np.int32)
        if bus.ndim == 1:
            bus = bus[:, None]
        bus = np.ascontiguousarray(bus)
        n, R = bus.shape
        g = None
        if gain is not None:
            g = np.ascontiguousarray(np.asarray(gain, dtype=np.float32).reshape(bus.shape))
        self._check(self.lib.oalsfx_engine_set_routes(self._h, int(first_stream), int(n), int(R), bus.ctypes.data,
                                                      None if g is None else g.ctypes.data, int(ramp_frames)))

    def set_bus_format(self, channel_format):
        """Every submix bus gets `channel_format` (a ChannelFormat; default: the engine's).  reduce_buses / mix_buses then
        write [n_buses][frames][bus_channels].  Refused while a pan route exists and the channel count would change."""
        self._check(self.lib.oalsfx_engine_set_bus_format(self._h, int(channel_format)))
        self.bus_format = int(channel_format)

    @property
    def bus_channels(self):
        """Channel count Cb of the submix buses."""
        return channel_count(self.bus_format)

    def set_route_pans(self, pan, bus, first_stream=0, ramp_frames=0):
        """Pan routes of streams first_stream, first_stream + 1, ...: bus[i] as in set_routes, each route with a
        [bus_channels][channels] matrix pan[i][r] (weight of stream channel k in bus channel j at [j][k]), its coefficients
        ramped from the route's current ones over ramp_frames frames.  `pan` is [n][R][Cb][C] with `bus` [n][R], or
        [n][Cb][C] with a 1-D `bus` (one route per stream)."""
        bus = np.asarray(bus, dtype=np.int32)
        if bus.ndim == 1:
            bus = bus[:, None]
        bus = np.ascontiguousarray(bus)
        n, R = bus.shape
        m = np.ascontiguousarray(np.asarray(pan, dtype=np.float32).reshape(n, R, self.bus_channels, self.channels))
        self._check(self.lib.oalsfx_engine_set_route_pans(self._h, int(first_stream), int(n), int(R), bus.ctypes.data,
                                                          m.ctypes.data, int(ramp_frames)))

    def _bus_count(self, frames, buses, n_buses):
        if n_buses is not None:
            return int(n_buses)
        size = buses.size if isinstance(buses, np.ndarray) else buses.numel() if hasattr(buses, "numel") else None
        if size is None:
            raise ValueError("n_buses is required for raw pointers")
        return size // (int(frames) * self.bus_channels)

    def reduce_buses(self, frames, dst, buses, layout=LAYOUT_STREAM_MAJOR, stream=0, n_buses=None):
        """buses ([n_buses][frames][bus_channels], device) = per bus the sum of the rows of `dst` (device, as mix() wrote it) of
        the active streams routed to it, in the fixed order of include/oalsfx_engine.h.  n_buses defaults to the size of
        `buses`."""
        self._check(self.lib.oalsfx_engine_reduce_buses(self._h, int(frames), _ptr(dst), layout,
                                                        self._bus_count(frames, buses, n_buses), _ptr(buses), C.c_void_p(stream)))
        return buses

    def mix_buses(self, src, dst, frames, buses, layout=LAYOUT_STREAM_MAJOR, stream=0, n_buses=None):
        """mix() on device buffers followed by reduce_buses() of its output on the same stream."""
        self._check(self.lib.oalsfx_engine_mix_buses(self._h, int(frames), _ptr(src), _ptr(dst), layout,
                                                     self._bus_count(frames, buses, n_buses), _ptr(buses), C.c_void_p(stream)))
        return buses

    def debug_state(self, stream, slot):
        out = (C.c_int32 * 4)()
        self._check(self.lib.oalsfx_engine_debug_state(self._h, stream, slot, out))
        return {"offset": out[0], "fade_count": out[1], "mod_index": out[2], "ring_mod_index": out[3]}

    def debug_waveshaper(self, samples, edge_coeff, out, count, stream=0):
        """The distortion stage's three waveshapers on a device buffer (test hook)."""
        self._check(self.lib.oalsfx_debug_waveshaper(self._h, _ptr(samples), float(edge_coeff), _ptr(out), int(count), stream))

    def pcm_to_float(self, src, bit_depth, dst, count, stream=0):
        """8/16-bit PCM -> float on device buffers (the reference demo's ingest, oalsfxpp_test.cpp:703-740)."""
        self._check(self.lib.oalsfx_pcm_to_float(self._h, _ptr(src), int(bit_depth), _ptr(dst), int(count),
                                                 C.c_void_p(stream)))
        return dst

    def float_to_s16(self, src, dst, rows, row_len, row_scale=None, stream=0):
        """float -> peak-normalised s16 per row on device buffers (the demo's egress, oalsfxpp_test.cpp:602-651)."""
        self._check(self.lib.oalsfx_float_to_s16(self._h, _ptr(src), _ptr(dst), int(rows), int(row_len),
                                                 _ptr(row_scale) if row_scale is not None else None, C.c_void_p(stream)))
        return dst

    def snapshot(self):
        """All stream state (delay lines, filter histories, pending flags) as one host byte array."""
        size = int(self.lib.oalsfx_engine_snapshot_size(self._h))
        buf = np.empty(size, dtype=np.uint8)
        self._check(self.lib.oalsfx_engine_snapshot(self._h, buf.ctypes.data, size))
        return buf

    def restore(self, snapshot):
        snapshot = np.ascontiguousarray(snapshot, dtype=np.uint8)
        self._check(self.lib.oalsfx_engine_restore(self._h, snapshot.ctypes.data, snapshot.size))

    _PLACEMENT = {"caller": 0, "auto": 1}

    def set_placement(self, mode):
        """"caller" (default: engine lane of stream s is s) or "auto": the engine moves streams between its lanes so
        that every 32-stream tile holds one parameter class.  Stream indices and buffers keep the caller's order."""
        if mode not in self._PLACEMENT:
            raise ValueError(f"placement must be one of {sorted(self._PLACEMENT)}")
        self._check(self.lib.oalsfx_engine_set_placement(self._h, self._PLACEMENT[mode]))

    @property
    def lane_of_stream(self):
        """The engine lane that holds each caller stream now (int32 array of num_streams)."""
        return self.lanes()[0]

    def lanes(self):
        """(lane_of_stream, the engine's lane count: a multiple of 32)."""
        out = np.empty(self.num_streams, dtype=np.int32)
        n = self.lib.oalsfx_engine_lanes(self._h, out.ctypes.data, self.num_streams)
        if n < 0:
            self._check(int(n))
        return out, int(n)

    @property
    def launch_count(self):
        return int(self.lib.oalsfx_engine_launch_count(self._h))

    @property
    def last_kernel(self):
        """Name of the mix kernel launched most recently (which kernel family served the last block)."""
        return self.lib.oalsfx_engine_last_kernel(self._h).decode()

    @property
    def device_bytes(self):
        return int(self.lib.oalsfx_engine_device_bytes(self._h))

"""numpy float32 model of routes with gains (include/oalsfx_engine.h, oalsfx_engine_set_routes).

A route is (stream, bus, g0, g1, Rf, T0).  Each route of an active stream becomes one virtual row gain(T) * x (one float32
rounding) with T = M + f; the virtual rows in stream-major order go through bus_model.model_buses, whose stable sort by bus
keeps ascending stream order inside each bus (a stream has at most one route per bus).  Routes replays the engine's
state on the host: the frame clock and every stream's routes."""
import numpy as np

from bus_model import model_buses

F32 = np.float32


def gain_at(g0, g1, rf, t0, t):
    """The header's expression in float32, one rounding per operation; arguments broadcast."""
    g0, g1 = np.asarray(g0, F32), np.asarray(g1, F32)
    rf, t0, t = np.asarray(rf, np.int64), np.asarray(t0, np.int64), np.asarray(t, np.int64)
    d = t - t0
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):   # (lanes the where below does not pick)
        ramp = g0 + (g1 - g0) * ((d + 1).astype(F32) / rf.astype(F32))
    return np.where(t < t0, g0, np.where((rf == 0) | (d >= rf), g1, ramp)).astype(F32)


class Routes:
    """Replays set_routes / route_streams / mix: routes[s] = {bus: (g0, g1, rf, t0)}.  A change without a ramp sets
    g0 = g1: it holds at once, also for a block mixed before it."""

    def __init__(self, S):
        self.routes = [{0: (F32(1), F32(1), 0, 0)} for _ in range(S)]
        self.clock = 0      # frames mixed so far
        self.M = 0          # clock at the start of the most recent mix

    def mixed(self, frames):
        self.M = self.clock
        self.clock += frames

    def set_routes(self, bus, gain=None, first_stream=0, ramp_frames=0):
        bus = np.asarray(bus, dtype=np.int32)
        if bus.ndim == 1:
            bus = bus[:, None]
        gain = np.ones(bus.shape, F32) if gain is None else np.asarray(gain, F32).reshape(bus.shape)
        t0 = self.clock
        for i in range(bus.shape[0]):
            old = self.routes[first_stream + i]
            new = {}
            for b, g in zip(bus[i].tolist(), gain[i]):
                if b >= 0:
                    g0 = g if ramp_frames == 0 else gain_at(*old[b], t0 - 1) if b in old else F32(0)
                    new[b] = (F32(g0), F32(g), int(ramp_frames), t0)
            self.routes[first_stream + i] = new

    def buses(self, rows, active, n_buses, M=None):
        """rows [S][frames][C] (caller order) -> [n_buses][frames][C], frame f at clock M + f (M: the last mix's)."""
        return model_routes(rows, self.routes, active, n_buses, self.M if M is None else M)


def model_routes(rows, routes, active, n_buses, M):
    rows = np.asarray(rows, dtype=F32)
    S, frames, C = rows.shape
    flat = [(s, b) + p for s in range(S) for b, p in routes[s].items()]
    if not flat:
        return np.zeros((n_buses, frames, C), F32)
    s, b, g0, g1, rf, t0 = (np.array(col) for col in zip(*flat))
    gains = gain_at(g0[:, None], g1[:, None], rf[:, None], t0[:, None], M + np.arange(frames)[None, :])
    with np.errstate(invalid="ignore"):    # 0 * Inf is NaN on the bus, as in the engine
        virt = gains[:, :, None] * rows[s]
    return model_buses(virt, b.astype(np.int32), np.asarray(active, bool)[s], n_buses)

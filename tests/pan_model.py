"""numpy float32 model of pan routes and bus formats (include/oalsfx_engine.h, oalsfx_engine_set_route_pans /
oalsfx_engine_set_bus_format), on top of route_model.

A route is (stream, bus) with either a gain (g0, g1) or a pan matrix pair (m0, m1) of [Cb][C], plus Rf and T0.  Each route of
an active stream becomes one virtual [frames][Cb] row: a scalar route's gain(T) * x_j in bus channel j < min(C, Cb) and +0.0f
above; a pan route's p = c_j0(T) * x_0, p = p + c_jk(T) * x_k, with every coefficient ramped by gain_at.  The virtual rows in
stream-major order go through bus_model.model_buses, as route_model's do."""
import numpy as np

from bus_model import model_buses
from route_model import gain_at

F32 = np.float32


def _diag(g, Cb, C):
    m = np.zeros((Cb, C), F32)
    for j in range(min(Cb, C)):
        m[j, j] = g
    return m


class Pans:
    """Replays set_routes / route_streams / set_route_pans / mix: routes[s] = {bus: ("g", g0, g1, rf, t0)} for a scalar
    route or {bus: ("p", m0, m1, rf, t0)} for a pan route."""

    def __init__(self, S, C, Cb=None):
        self.C, self.Cb = C, C if Cb is None else Cb
        self.routes = [{0: ("g", F32(1), F32(1), 0, 0)} for _ in range(S)]
        self.clock = 0
        self.M = 0

    def mixed(self, frames):
        self.M = self.clock
        self.clock += frames

    def _at(self, route, t):
        """A route's matrix at clock t ([Cb][C]: a scalar route's gain on the index diagonal)."""
        kind, a0, a1, rf, t0 = route
        if kind == "g":
            return _diag(gain_at(a0, a1, rf, t0, t), self.Cb, self.C)
        return gain_at(a0, a1, rf, t0, t)

    def _set(self, bus, target, first_stream, ramp_frames, pan):
        bus = np.asarray(bus, dtype=np.int32)
        if bus.ndim == 1:
            bus = bus[:, None]
        t0 = self.clock
        for i in range(bus.shape[0]):
            old = self.routes[first_stream + i]
            new = {}
            for r, b in enumerate(bus[i].tolist()):
                if b < 0:
                    continue
                prev = old.get(b)
                if not pan and not (prev is not None and prev[0] == "p" and ramp_frames > 0):
                    g1 = F32(target[i][r])
                    g0 = g1 if ramp_frames == 0 else gain_at(*prev[1:], t0 - 1) if prev is not None else F32(0)
                    new[b] = ("g", F32(g0), g1, int(ramp_frames), t0)
                    continue
                m1 = np.asarray(target[i][r], F32).reshape(self.Cb, self.C) if pan else _diag(target[i][r], self.Cb, self.C)
                if ramp_frames == 0:
                    m0 = m1.copy()
                elif prev is not None:
                    m0 = self._at(prev, t0 - 1)
                else:
                    m0 = np.zeros((self.Cb, self.C), F32)
                new[b] = ("p", m0, m1, int(ramp_frames), t0)
            self.routes[first_stream + i] = new

    def set_routes(self, bus, gain=None, first_stream=0, ramp_frames=0):
        shape = np.asarray(bus).reshape(len(bus), -1).shape
        gain = np.ones(shape, F32) if gain is None else np.asarray(gain, F32).reshape(shape)
        self._set(bus, gain, first_stream, ramp_frames, pan=False)

    def set_route_pans(self, pan, bus, first_stream=0, ramp_frames=0):
        shape = np.asarray(bus).reshape(len(bus), -1).shape
        self._set(bus, np.asarray(pan, F32).reshape(shape + (self.Cb, self.C)), first_stream, ramp_frames, pan=True)

    def buses(self, rows, active, n_buses, M=None):
        """rows [S][frames][C] (caller order) -> [n_buses][frames][Cb], frame f at clock M + f (M: the last mix's)."""
        return model_pans(rows, self.routes, active, n_buses, self.M if M is None else M, self.Cb)


def _virtual_rows(routes, x, T, Cb):
    """[n][frames][Cb] member values of n routes of one kind for their rows x [n][frames][C] at clock values T [frames]."""
    kind = routes[0][0]
    a0, a1 = np.stack([r[1] for r in routes]).astype(F32), np.stack([r[2] for r in routes]).astype(F32)
    rf, t0 = np.array([r[3] for r in routes], np.int64), np.array([r[4] for r in routes], np.int64)
    n, frames, C = x.shape
    with np.errstate(invalid="ignore", over="ignore"):    # 0 * Inf is NaN on the bus, as in the engine
        if kind == "g":
            g = gain_at(a0[:, None], a1[:, None], rf[:, None], t0[:, None], T[None, :])
            out = np.zeros((n, frames, Cb), F32)
            for j in range(min(C, Cb)):
                out[:, :, j] = g * x[:, :, j]
            return out
        c = gain_at(a0[:, None], a1[:, None], rf[:, None, None, None], t0[:, None, None, None], T[None, :, None, None])
        p = c[..., 0] * x[:, :, None, 0]
        for k in range(1, C):
            p = p + c[..., k] * x[:, :, None, k]
        return p.astype(F32)


def model_pans(rows, routes, active, n_buses, M, Cb):
    rows = np.asarray(rows, dtype=F32)
    S, frames, C = rows.shape
    batch = max(1, (1 << 24) // (frames * Cb * C))     # routes per pass: bounds the [routes][frames][Cb][C] coefficients
    T = M + np.arange(frames, dtype=np.int64)
    flat = [(s, b, route) for s in range(S) for b, route in routes[s].items()]
    if not flat:
        return np.zeros((n_buses, frames, Cb), F32)
    virt = np.empty((len(flat), frames, Cb), F32)
    for kind in ("g", "p"):
        idx = [i for i, f in enumerate(flat) if f[2][0] == kind]
        for q in range(0, len(idx), batch):
            part = idx[q:q + batch]
            virt[part] = _virtual_rows([flat[i][2] for i in part], rows[[flat[i][0] for i in part]], T, Cb)
    s = np.array([f[0] for f in flat])
    b = np.array([f[1] for f in flat], np.int32)
    return model_buses(virt, b, np.asarray(active, bool)[s], n_buses)

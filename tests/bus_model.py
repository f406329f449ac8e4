"""numpy float32 model of the submix buses' summation order (include/oalsfx_engine.h, oalsfx_engine_reduce_buses).

Bus b's members -- the active streams routed to it -- in ascending stream index are the level-0 list.  Each level is padded
to a multiple of 32 entries with +0.0f and summed in runs of 32 by 32 explicit sequential float32 additions from +0.0f;
the run sums are the next level's list, until one entry is left.  No np.sum: its pairwise order is not the contract."""
import numpy as np

RUN = 32


def bus_members(routing, active, n_buses):
    routing = np.asarray(routing)
    live = np.flatnonzero(np.asarray(active, dtype=bool) & (routing >= 0))
    order = live[np.argsort(routing[live], kind="stable")]      # by bus, ascending stream index inside a bus
    return np.split(order, np.cumsum(np.bincount(routing[order], minlength=n_buses))[:-1])


def model_buses(rows, routing, active, n_buses):
    """rows: [S][frames][C] float32 (caller stream order).  Returns [n_buses][frames][C] float32."""
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    S, frames, C = rows.shape
    flat = np.concatenate([rows.reshape(S, frames * C), np.zeros((1, frames * C), np.float32)])   # row S: the +0.0f pad
    lists = [(b, m) for b, m in enumerate(bus_members(routing, active, n_buses))]
    out = np.zeros((n_buses, frames * C), np.float32)
    level_rows = flat
    while lists:
        # every open list padded to whole runs: idx[r][i] = the row of entry i of run r, or the zero row
        idx, owner = [], []
        for b, m in lists:
            n_runs = max(1, -(-len(m) // RUN))
            padded = np.full(n_runs * RUN, level_rows.shape[0] - 1, dtype=np.int64)
            padded[:len(m)] = m
            idx.append(padded.reshape(n_runs, RUN))
            owner.append((b, n_runs))
        idx = np.concatenate(idx)
        acc = np.zeros((idx.shape[0], frames * C), np.float32)
        for i in range(RUN):
            acc = acc + level_rows[idx[:, i]]
        nxt, first = [], 0
        for b, n_runs in owner:
            if n_runs == 1:
                out[b] = acc[first]
            else:
                nxt.append((b, np.arange(first, first + n_runs)))
            first += n_runs
        level_rows = np.concatenate([acc, np.zeros((1, frames * C), np.float32)])
        lists = nxt
    return out.reshape(n_buses, frames, C)

"""CPU statement of the device-kept per-bearer byte FIFOs (rs_enable_buffers, include/rs_sched.h), test-only.

Each bearer holds at most K records (arrival time, bytes), `queued` (their sum) and `dropped`; a backlogged bearer has
no FIFO.  At every TTI: (1) the arrival is pushed, or dropped whole when K records are held; (2) the scheduler is shown
queue min(queued, INT32_MAX) and HoL now - head arrival time (0 when empty; 100000000 / 0 for a backlogged bearer);
(3) the TTI is scheduled; (4) the bytes booked to the bearer, clamped to queued, leave from the head, and a record sent
in part keeps its arrival time.  :func:`closed_loop` drives the oracle (or a non-buffered CUDA handle) through that
loop one TTI at a time with ``step(queue=, hol=)`` and takes the departures from its cum_bytes deltas."""
from __future__ import annotations

import numpy as np

INFINITE = 100000000
INT32_MAX = 2147483647


class BufferModel:
    def __init__(self, shape, max_records, backlogged=None):
        self.shape = tuple(shape)
        self.K = int(max_records)
        n = int(np.prod(self.shape))
        self.backlogged = np.zeros(n, bool) if backlogged is None else np.asarray(backlogged, bool).reshape(n).copy()
        self.fifo = [[] for _ in range(n)]   # [[arrival_time, bytes], ...], head first
        self.queued = np.zeros(n, np.int64)
        self.dropped = np.zeros(n, np.uint64)

    def arrive(self, arrivals, now, arrival_time):
        """Steps 1-2 of one TTI; returns the (queue int32, hol float64) the scheduler sees, shaped like the bearers."""
        a = np.asarray(arrivals).reshape(-1)
        q = np.empty(a.shape[0], np.int32)
        h = np.empty(a.shape[0], np.float64)
        now, at = float(now), float(arrival_time)
        for i in range(a.shape[0]):
            if self.backlogged[i]:
                q[i], h[i] = INFINITE, 0.0
                continue
            f = self.fifo[i]
            if a[i] > 0:
                if len(f) == self.K:
                    self.dropped[i] += np.uint64(a[i])
                else:
                    f.append([at, int(a[i])])
                    self.queued[i] += int(a[i])
            q[i] = min(int(self.queued[i]), INT32_MAX)
            h[i] = now - f[0][0] if f else 0.0
        return q.reshape(self.shape), h.reshape(self.shape)

    def depart(self, booked):
        """Step 4: booked = bytes credited to each bearer this TTI (its cum_bytes increment)."""
        b = np.asarray(booked, dtype=np.int64).reshape(-1)
        for i in np.flatnonzero(b > 0):
            if self.backlogged[i]:
                continue
            left = min(int(b[i]), int(self.queued[i]))
            self.queued[i] -= left
            f = self.fifo[i]
            while left > 0:
                if f[0][1] > left:
                    f[0][1] -= left
                    break
                left -= f.pop(0)[1]

    def state(self):
        """What rs_get_buffers returns (a backlogged bearer reports 0 everywhere)."""
        n = len(self.fifo)
        st = {"queued": np.where(self.backlogged, 0, self.queued).astype(np.int64),
              "n_records": np.array([0 if self.backlogged[i] else len(self.fifo[i]) for i in range(n)], np.int32),
              "head_time": np.array([self.fifo[i][0][0] if self.fifo[i] and not self.backlogged[i] else 0.0
                                     for i in range(n)], np.float64),
              "dropped": np.where(self.backlogged, 0, self.dropped).astype(np.uint64)}
        return {k: v.reshape(self.shape) for k, v in st.items()}


def closed_loop(sched, model, cqi, draws, dts, arrivals, now, arrival_time, active=None, bounds=(), want_aux=True):
    """Run T TTIs through `sched` (OracleScheduler, or a CUDA Scheduler without buffers) one step per TTI with the queue
    state from `model`.  Returns (outputs [T][B][...] incl. queue_out / hol_out, scheduler states and buffer states after
    the TTIs in `bounds`)."""
    outs, states, bufs = [], [], []
    for t in range(len(dts)):
        q, h = model.arrive(arrivals[t], now[t], arrival_time[t])
        before = sched.get_state()["cum_bytes"].astype(np.int64)
        o = sched.step(cqi[t], draws[t], dt=float(dts[t]), active=None if active is None else active[t],
                       want_aux=want_aux, queue=q, hol=h)
        after = sched.get_state()
        model.depart(after["cum_bytes"].astype(np.int64) - before)
        o["queue_out"], o["hol_out"] = q, h
        outs.append(o)
        if t + 1 in bounds:
            states.append(after)
            bufs.append(model.state())
    return {k: np.stack([x[k] for x in outs]) for k in outs[0]}, states, bufs

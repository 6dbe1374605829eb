"""GPU: histograms of per-UE throughput over active time (rs_enable_ue_upt_hist / rs_get_ue_upt_hist /
rs_ue_upt_hist_device / rs_reduce_ue_upt_hist, rs_batch --upt-bin-bytes), tolerance 0: the device counts equal
workload.ue_upt_hist fed the run's own queue_out and the cum_bytes get_state returns at the windows' ends, for every id,
every run entry point with and without the caller's queue_out, split batches, device-drawn traffic, profiles and the
restart and switch-off rules; one case checked against the buffer model's drain time instead of the twin."""
import ctypes as C

import numpy as np
import pytest

from oracle.pyoracle import OracleScheduler
from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import SRC_NONE, SRC_ONOFF, SRC_PERIODIC, SRC_RATE
from tests import test_rs_batch_buffers_gpu as rbb
from tests.buffer_model import BufferModel, closed_loop
from tests.test_buffers_gpu import K, Traffic
from tests.test_channel_gpu import COUNTS
from tests.test_host_api_gpu import _nccl
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu
BINS, BIN_BYTES = 40, 300            # UPT: bytes per active TTI
RATE_BINS, RATE_BYTES = 30, 4000     # the throughput histogram whose windows UPT uses
HOL_BINS = 24


def _torch(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cum(g):
    return g.get_state()["cum_bytes"]


def _handle(c, tr, P=1, hol=False):
    """A buffered handle of Case c (P profiles: rolled slice maps, cell b on profile b % P) with the throughput and UPT
    histograms on (and the HoL histogram with hol); returns (handle, u2s [P][U], cell_profile)."""
    if P == 1:
        g, u2s, cp = c.scheduler(), c.u2s[None], None
    else:
        u2s = np.stack([np.roll(c.u2s, 3 * p) for p in range(P)])
        cp = np.arange(c.B) % P
        g = sched.Scheduler.from_profiles(c.algo, [(c.w, c.p, m) for m in u2s], cp.astype(np.int32), **c.cfg())
        if c.trace:
            g.set_traces(c.traces, c.ue_trace)
    g.enable_buffers(K, tr.backlogged)
    if hol:
        g.enable_hol_hist(HOL_BINS)
    g.enable_ue_rate_hist(RATE_BINS, RATE_BYTES)
    g.enable_ue_upt_hist(BINS, BIN_BYTES)
    return g, u2s, cp


class Runner:
    """TTIs [t0, t1) of Case c with Traffic tr through one entry point (rs_step: one call per TTI); with_out False: no
    queue_out, so the handle's own scratch (rs_run_device) or slot ring (host calls) feeds the active counts.
    span() returns the queues the TTIs showed, [n][B][U](, 2), or None; `close` runs after the call's enqueue (before
    rs_wait / the synchronisation)."""

    def __init__(self, c, tr, entry, tpl=16, with_out=True):
        self.c, self.tr, self.entry, self.tpl, self.with_out = c, tr, entry, tpl, with_out
        if entry in ("run_device", "run_traces_device"):
            self.d_arr, self.d_draws = _torch(tr.arr), _torch(c.draws)
            self.d_cqi = None if c.trace else _torch(c.slabs)

    def span(self, g, t0, t1, close=False):
        if self.entry in ("run_device", "run_traces_device"):
            return self._device(g, t0, t1, close)
        qs = [self._host(g, t, t + 1, close and t == t1 - 1) for t in range(t0, t1)] if self.entry == "step" else \
            [self._host(g, t0, t1, close)]
        return np.concatenate(qs) if self.with_out else None

    def _host(self, g, t0, t1, close):
        c, tr, L, n, sl = self.c, self.tr, sched.lib(), t1 - t0, slice(t0, t1)
        step = self.entry == "step"
        out, o = g._host_outputs(None if step else n, False)
        arr = np.ascontiguousarray(tr.arr[sl], dtype=np.int32)
        nw, at = np.ascontiguousarray(c.now[sl]), np.ascontiguousarray(tr.at[sl])
        qo = np.zeros(arr.shape, np.int32) if self.with_out else None
        ho = np.zeros(arr.shape, np.float64) if self.with_out else None
        tf = sched._Traffic(sched._ptr(arr), sched._ptr(nw), sched._ptr(at), sched._ptr(qo), sched._ptr(ho))
        sched._check(L.rs_set_traffic(g._h, C.byref(tf)))
        draws = np.ascontiguousarray(c.draws[t0] if step else c.draws[sl])
        dt = np.ascontiguousarray(c.dts[sl])
        ticket = C.c_int64(-1)
        if step:
            rc = L.rs_step(g._h, sched._ptr(np.ascontiguousarray(c.slabs[t0])), sched._ptr(draws), None, float(dt[0]),
                           C.byref(o))
        elif self.entry in ("run_host", "run_host_async"):
            args = [g._h, n, sched._ptr(np.ascontiguousarray(c.slabs[sl])), 1, sched._ptr(draws), None, sched._ptr(dt),
                    C.byref(o), self.tpl]
            rc = L.rs_run_host(*args) if self.entry == "run_host" else L.rs_run_host_async(*args, C.byref(ticket))
        else:
            args = [g._h, n, sched._ptr(np.ascontiguousarray(c.rows[sl])), sched._ptr(draws), None, sched._ptr(dt),
                    C.byref(o), self.tpl]
            rc = L.rs_run_traces_host(*args) if self.entry == "run_traces_host" else \
                L.rs_run_traces_host_async(*args, C.byref(ticket))
        sched._check(rc)
        if close:
            g.close_ue_rate_window()   # an async call's kernels may still run: the close is ordered after them
        if ticket.value >= 0:
            g.wait(ticket.value)
        del out
        return qo

    def _device(self, g, t0, t1, close):
        import torch
        c, tr, n, sl = self.c, self.tr, t1 - t0, slice(t0, t1)
        d_q = torch.zeros((n,) + tr.arr.shape[1:], dtype=torch.int32, device="cuda") if self.with_out else None
        kw = dict(ttis_per_launch=self.tpl, d_arrivals=self.d_arr[t0].data_ptr(), now=c.now[sl], arrival_time=tr.at[sl],
                  d_queue_out=d_q.data_ptr() if self.with_out else 0)
        if self.entry == "run_device":
            g.run_device(n, self.d_cqi[t0].data_ptr(), c.B * c.U * c.G, self.d_draws[t0].data_ptr(), c.dts[sl], **kw)
        else:
            g.run_traces_device(n, c.rows[sl], self.d_draws[t0].data_ptr(), c.dts[sl], **kw)
        if close:
            g.close_ue_rate_window()
        g.sync()
        return d_q.cpu().numpy() if self.with_out else None


def _windows(T, n):
    edges = np.linspace(0, T, n + 1).astype(int)
    return [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:])]


def _run_windows(c, g, run, windows, u2s, cp):
    """Run and close the windows; returns (device UPT counts, twin of the run's own queues, device rate counts, rate
    twin).  Without queue_out the UPT twin stays zero."""
    want = np.zeros((u2s.shape[0], c.S, BINS), np.uint64)
    want_rate = np.zeros((u2s.shape[0], c.S, RATE_BINS), np.uint64)
    prev = _cum(g)
    for t0, t1 in windows:
        q = run.span(g, t0, t1, close=True)
        cur = _cum(g)
        if q is not None:
            want += workload.ue_upt_hist(q, prev, cur, u2s, c.S, BINS, BIN_BYTES, cp)
        want_rate += workload.ue_rate_hist(prev, cur, u2s, c.S, RATE_BINS, RATE_BYTES, cp)
        prev = cur
    return g.get_ue_upt_hist(), want, g.get_ue_rate_hist(), want_rate


def _spread(want):
    """Samples in at least three bins."""
    return np.count_nonzero(want.sum(axis=(0, 1))) >= 3


def _check_entry(algo, nb, P, entry, tpl=16, T=40, B=9, n_windows=3, seed=0):
    """The same run with and without the caller's queue_out: both counts equal the twin of the first run's queues."""
    trace = "traces" in entry
    c = Case(algo, CELLS["narrow"], B=B, T=T, seed=9100 + algo + 10 * nb + P + seed, trace=trace, nb=nb, active=False)
    tr = Traffic(c, seed=algo + nb + P + seed)
    got = []
    for with_out in (True, False):
        g, u2s, cp = _handle(c, tr, P)
        h, w, r, wr = _run_windows(c, g, Runner(c, tr, entry, tpl, with_out), _windows(T, n_windows), u2s, cp)
        if with_out:
            want = w
        assert np.array_equal(r, wr), entry   # the throughput histogram is as before
        got.append(h)
        g.close()
    assert got[0].shape == (P, c.S, BINS)
    assert np.array_equal(got[0], want), entry
    assert np.array_equal(got[1], want), entry + " (scratch)"
    assert _spread(want)
    return want


@pytest.mark.parametrize("algo", IDS)
def test_every_id_equals_twin(algo):
    _check_entry(algo, 1 if algo == 1 else 2, 1, "run_device")


ENTRIES = ["step", "run_host", "run_host_async", "run_traces_host", "run_traces_host_async", "run_device",
           "run_traces_device"]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("nb", [1, 2])
def test_every_entry_point_equals_twin(entry, nb):
    _check_entry(9 if nb == 2 else 8, nb, 1, entry, T=24 if entry == "step" else 40)


@pytest.mark.parametrize("entry", ["run_device", "run_host"])
@pytest.mark.parametrize("tpl", [1, 16, 64])
def test_ttis_per_launch_and_windows_over_several_launches(entry, tpl):
    _check_entry(10, 2, 1, entry, tpl=tpl, T=70, n_windows=2, seed=tpl)


@pytest.mark.parametrize("entry", ["run_device", "run_host"])
def test_batch_split_over_streams(entry):
    """2400 narrow cells: the handle runs its batch as two parts on two streams, each part counting its own cells."""
    _check_entry(9, 2, 1, entry, tpl=8, T=40, B=2400, n_windows=2)


def test_three_profiles_moved_between_windows():
    """rs_set_cell_profiles between windows: later samples go to each cell's new profile and its slices; the active
    counts of the open window are kept."""
    c = Case(9, CELLS["narrow"], B=12, T=45, seed=9400, nb=2, active=False)
    tr = Traffic(c, seed=5)
    g, u2s, cp = _handle(c, tr, 3)
    run = Runner(c, tr, "run_host")
    want = np.zeros((3, c.S, BINS), np.uint64)
    prev, qs = _cum(g), []
    for k, (t0, t1) in enumerate(_windows(c.T, 3)):
        mid = (t0 + t1) // 2
        qs.append(run.span(g, t0, mid))
        if k:
            cp = (cp + 1 + k) % 3   # mid-window
            g.set_cell_profiles(cp.astype(np.int32))
        qs.append(run.span(g, mid, t1, close=True))
        cur = _cum(g)
        want += workload.ue_upt_hist(np.concatenate(qs), prev, cur, u2s, c.S, BINS, BIN_BYTES, cp)
        prev, qs = cur, []
    got = g.get_ue_upt_hist()
    g.close()
    assert got.shape == (3, c.S, BINS) and np.array_equal(got, want)
    assert all(want[p].sum() > 0 for p in range(3)) and _spread(want)


def test_device_drawn_traffic_and_channel():
    """rs_synth_traffic (RATE, PERIODIC, ONOFF and backlogged slices) and rs_synth_channel (fading and i.i.d. slices),
    the HoL histogram on as well."""
    import torch
    c = Case(9, CELLS["narrow"], B=11, T=60, seed=9500, nb=2, active=False)
    on, off = sched.onoff_spec(5, 8)
    kinds = [{"kind": SRC_NONE}, {"kind": SRC_PERIODIC, "period_ttis": 5, "frame_bytes": [20000, 3000, 7000]},
             {"kind": SRC_ONOFF, "pkt_bytes": 900, "period_ttis": 2, "leave_on_q32": on, "leave_off_q32": off},
             {"kind": SRC_RATE, "pkt_bytes": 1500, "pkts_q16": sched.arrival_spec(1500, 4.0)[1]}]
    tr = Traffic(c, seed=1)
    tr.backlogged[:] = (c.u2s % 4 == 0)[None, :, None]
    g, u2s, _ = _handle(c, tr, hol=True)
    g.set_sources([kinds[s % 4] for s in range(c.S)])
    g.set_channels([sched.channel_spec(COUNTS, 1.5, 6, 4) if s % 2 else {"kind": workload.CH_IID} for s in range(c.S)])
    per = (c.T, c.B, c.U, 2)
    d_arr = torch.zeros(per, dtype=torch.int32, device="cuda")
    d_q = torch.zeros(per, dtype=torch.int32, device="cuda")
    d_cqi = torch.zeros((c.T, c.B, c.U, c.G), dtype=torch.uint8, device="cuda")
    g.synth_traffic(5, 0, 0, c.T, d_arr.data_ptr())
    g.synth_channel(5, 0, 0, c.T, d_cqi.data_ptr())
    d_draws = _torch(c.draws)
    want = np.zeros((1, c.S, BINS), np.uint64)
    prev = _cum(g)
    for t0, t1 in _windows(c.T, 3):
        g.run_device(t1 - t0, d_cqi[t0].data_ptr(), d_cqi[0].numel(), d_draws[t0].data_ptr(), c.dts[t0:t1],
                     ttis_per_launch=16, d_arrivals=d_arr[t0].data_ptr(), now=c.now[t0:t1], arrival_time=tr.at[t0:t1],
                     d_queue_out=d_q[t0].data_ptr())
        g.close_ue_rate_window()
        cur = _cum(g)
        want += workload.ue_upt_hist(d_q[t0:t1].cpu().numpy(), prev, cur, u2s, c.S, BINS, BIN_BYTES)
        prev = cur
    got = g.get_ue_upt_hist()
    assert g.get_hol_hist().sum() > 0
    g.close()
    assert np.array_equal(got, want) and _spread(want)
    assert want[0, 1::4].sum() > 0 and want[0, 2::4].sum() > 0   # PERIODIC and ONOFF slices have samples


def test_back_to_back_closes_add_no_samples():
    c = Case(8, CELLS["narrow"], B=5, T=20, seed=9700, active=False)
    tr = Traffic(c, seed=2)
    g, u2s, cp = _handle(c, tr)
    g.close_ue_rate_window()   # right after enabling: no active TTI yet
    assert not g.get_ue_upt_hist().any()
    got, want, _, _ = _run_windows(c, g, Runner(c, tr, "run_device"), [(0, 20)], u2s, cp)
    g.close_ue_rate_window()
    g.close_ue_rate_window()
    assert np.array_equal(g.get_ue_upt_hist(), want) and np.array_equal(got, want) and want.sum() > 0
    assert g.get_ue_rate_hist()[0, :, 0].sum() >= 2 * c.B * c.U   # the throughput histogram's bin-0 samples
    g.close()


@pytest.mark.parametrize("nb", [1, 2])
def test_restarts(nb):
    """Mid-window: rs_enable_ue_upt_hist (restarts both windows, adds and clears no throughput samples), rs_set_state
    with counters below 2^32 and near 2^64, rs_reset_state; each zeroes the active counts with its snapshot change, and
    the restarted window matches the twin from there."""
    c = Case(9 if nb == 2 else 10, CELLS["narrow"], B=8, T=60, seed=9600 + nb, nb=nb, active=False)
    tr = Traffic(c, seed=nb)
    g, u2s, _ = _handle(c, tr)
    run = Runner(c, tr, "run_device" if nb == 2 else "run_host")
    rng = np.random.default_rng(nb)
    shape = tr.backlogged.shape
    want = np.zeros((1, c.S, BINS), np.uint64)
    want_rate = np.zeros((1, c.S, RATE_BINS), np.uint64)
    prev = _cum(g)
    for k, (t0, t1) in enumerate(_windows(c.T, 5)):
        if k:   # the TTIs of the window so far are dropped with the old counts
            run.span(g, t0, t0 + 3)
            t0 += 3
            if k == 1:
                before = g.get_ue_rate_hist()
                g.enable_ue_upt_hist(BINS, BIN_BYTES)
                assert np.array_equal(g.get_ue_rate_hist(), before) and not g.get_ue_upt_hist().any()
                want[:] = 0
                prev = _cum(g)
            elif k in (2, 3):
                base = (1 << 32) - 20000 if k == 2 else (1 << 64) - 20000
                prev = (np.uint64(base) + rng.integers(0, 15000, shape).astype(np.uint64)).astype(np.uint64)
                g.set_state(cum_bytes=prev)
            else:
                g.reset_state()
                prev = np.zeros(shape, np.uint64)
        q = run.span(g, t0, t1, close=True)
        cur = _cum(g)
        if k == 3:
            assert (cur < prev).any()   # some counters wrapped past 2^64 in this window
        want += workload.ue_upt_hist(q, prev, cur, u2s, c.S, BINS, BIN_BYTES)
        want_rate += workload.ue_rate_hist(prev, cur, u2s, c.S, RATE_BINS, RATE_BYTES)
        prev = cur
    got, rate = g.get_ue_upt_hist(), g.get_ue_rate_hist()
    g.close()
    assert np.array_equal(got, want) and _spread(want)
    assert np.array_equal(rate, want_rate)
    assert want.sum() < 4 * c.B * c.U   # some UEs had no data queued in some windows


def test_switching_off_and_refusals():
    import torch
    c = Case(9, CELLS["narrow"], B=5, T=30, seed=9800, nb=2, active=False)
    tr = Traffic(c, seed=6)
    g = c.scheduler()
    with pytest.raises(sched.RsError, match="no UPT histogram"):
        g.get_ue_upt_hist()
    with pytest.raises(sched.RsError, match="no buffers"):
        g.enable_ue_upt_hist(4, 100)
    g.enable_buffers(K, tr.backlogged)
    with pytest.raises(sched.RsError, match="no throughput histogram"):
        g.enable_ue_upt_hist(4, 100)
    g.enable_ue_rate_hist(RATE_BINS, RATE_BYTES)
    for n, x, what in [(-1, 100, "n_bins -1 outside 0..65536"), (65537, 100, "n_bins 65537"),
                       (4, 0, "bin_bytes 0 is not >= 1"), (4, -7, "bin_bytes -7")]:
        with pytest.raises(sched.RsError, match=what):
            g.enable_ue_upt_hist(n, x)
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == 0
    g.enable_ue_upt_hist(BINS, BIN_BYTES)
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == BINS
    got, want, _, _ = _run_windows(c, g, Runner(c, tr, "run_device"), [(0, 15)], c.u2s[None], None)
    assert np.array_equal(got, want) and want.sum() > 0
    d = torch.full((c.S * BINS,), 7, dtype=torch.int64, device="cuda")
    g.ue_upt_hist_device(d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64).reshape(got.shape), got)
    g.set_cell_profiles(np.zeros(c.B, np.int32))   # leaves it on
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == BINS
    g.enable_ue_rate_hist(RATE_BINS, RATE_BYTES)   # replaces the windows: off
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == 0
    with pytest.raises(sched.RsError, match="rs_get_ue_upt_hist: the handle has no UPT histogram"):
        g.get_ue_upt_hist()
    g.enable_ue_upt_hist(BINS, BIN_BYTES)
    g.enable_buffers(K, tr.backlogged)             # the buffers again: off
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == 0
    g.enable_ue_upt_hist(BINS, BIN_BYTES)
    g.enable_ue_upt_hist(0, 0)                     # off and freed
    with pytest.raises(sched.RsError, match="rs_ue_upt_hist_device: the handle has no UPT histogram"):
        g.ue_upt_hist_device(d.data_ptr())
    g.enable_ue_upt_hist(BINS, BIN_BYTES)
    g.enable_buffers(0)
    assert sched.lib().rs_ue_upt_hist_bins(g._h) == 0
    g.close()
    S = 64   # 65 profiles x 64 slices x 65536 bins of uint64: 2080 MiB
    u2s = np.repeat(np.arange(S), 2).astype(np.int32)
    big = sched.Scheduler.from_profiles(9, [(np.full(S, 1 / S), np.tile(c.p[:1], (S, 1)), u2s)] * 65,
                                        np.arange(65, dtype=np.int32))
    big.enable_buffers(2)
    big.enable_ue_rate_hist(1, 1)
    with pytest.raises(sched.RsError, match="exceed 2 GiB"):
        big.enable_ue_upt_hist(65536, 1)
    big.enable_ue_upt_hist(16384, 1)
    big.close()


def test_one_arrival_lands_on_the_bin_of_its_drain_time():
    """One cell, one UE with a FIFO, one arrival of X bytes at TTI 0, fixed CQI: its one sample is X / k bytes per TTI,
    k the TTIs the buffer model (driving the CPU oracle) takes to drain it."""
    X, T, bin_bytes = 150000, 40, 100
    u2s = np.zeros(1, np.int32)
    w, p = np.ones(1), np.array([[0, 0, 1, 1]], np.int32)
    cqi = np.full((T, 1, 1, 64), 9, np.uint8)
    draws = workload.synth_rand_draws(3, 0, 1, 0, T, 1, 2)
    now, dts = workload.tti_clock(T)
    arr = np.zeros((T, 1, 1), np.int32)
    arr[0, 0, 0] = X
    at = now - 0.0005
    o = OracleScheduler(9, w, p, u2s, 1)
    outs, _, _ = closed_loop(o, BufferModel((1, 1), K), cqi, draws, dts, arr, now, at)
    k = int((outs["queue_out"] > 0).sum())
    assert 2 <= k < T and outs["queue_out"][-1].sum() == 0
    g = sched.Scheduler(9, w, p, u2s, 1)
    g.enable_buffers(K)
    g.enable_ue_rate_hist(10, 1)
    g.enable_ue_upt_hist(4000, bin_bytes)
    g.run_host(cqi, draws, dts, arrivals=arr, now=now, arrival_time=at)
    g.close_ue_rate_window()
    h = g.get_ue_upt_hist()
    g.close()
    assert int(_cum_sum(o)) == X   # every byte booked once
    assert h.sum() == 1 and h[0, 0, X // k // bin_bytes] == 1, (k, np.flatnonzero(h))


def _cum_sum(o):
    return o.get_state()["cum_bytes"].astype(np.int64).sum()


def test_schedules_state_buffers_and_histograms_do_not_change():
    """A split buffered batch through rs_run_device and a host run: every output, the state, the buffers, the HoL and
    the throughput histograms are the same bits with UPT on and off."""
    from tests.test_hol_hist_gpu import _handle as hol_handle, _run
    for entry, B, T in (("run_device", 2400, 20), ("run_host", 7, 33)):
        c = Case(10, CELLS["narrow"], B=B, T=T, seed=9750, nb=2, active=False)
        tr = Traffic(c, seed=3)
        runs = []
        for on in (True, False):
            g, _, _ = hol_handle(c, tr, 1)
            g.enable_ue_rate_hist(RATE_BINS, RATE_BYTES)
            if on:
                g.enable_ue_upt_hist(BINS, BIN_BYTES)
            res = _run(c, g, tr, entry, 16, True)
            g.close_ue_rate_window()
            if on:
                assert g.get_ue_upt_hist().sum() > 0
            runs.append((res, g.get_state(), g.get_buffers(), g.get_stats(), g.get_buffer_stats(), g.get_hol_hist(),
                         g.get_ue_rate_hist()))
            g.close()
        (r0, s0, b0, *x0), (r1, s1, b1, *x1) = runs
        for x, y in zip(r0, r1):
            assert np.array_equal(x, y), entry
        for d0, d1 in ((s0, s1), (b0, b1)):
            for k in d0:
                assert np.array_equal(d0[k], d1[k]), (entry, k)
        assert all(np.array_equal(x, y) for x, y in zip(x0, x1)), entry


def test_single_rank_reduce_equals_get():
    c = Case(9, CELLS["narrow"], B=6, T=40, seed=9900, nb=2, active=False)
    tr = Traffic(c, seed=4, n_profiles=2, cell_profile=np.arange(c.B) % 2)
    g, u2s, cp = _handle(c, tr, 2)
    _run_windows(c, g, Runner(c, tr, "run_device", with_out=False), _windows(c.T, 2), u2s, cp)
    L = _nccl()
    L.rs_reduce_ue_upt_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    uid = (C.c_uint8 * 128)()
    assert L.rs_comm_unique_id(uid) == 0, L.rs_nccl_last_error()
    comm = C.c_void_p()
    assert L.rs_comm_init_rank(1, 0, uid, 0, C.byref(comm)) == 0, L.rs_nccl_last_error()
    red = np.zeros((2, c.S, BINS), dtype=np.uint64)
    assert L.rs_reduce_ue_upt_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, L.rs_nccl_last_error()
    assert np.array_equal(red, g.get_ue_upt_hist()) and red.sum() > 0
    g.enable_ue_upt_hist(0, 0)
    assert L.rs_reduce_ue_upt_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) != 0
    assert b"rs_ue_upt_hist_device" in L.rs_nccl_last_error()
    L.rs_comm_destroy(comm)
    g.close()


# ---- rs_batch --upt-bin-bytes ------------------------------------------------------------------------------------------
def _batch_mirror(algo, cfgs, trafs, B, T, seed, W, n_bins, upt_bytes):
    """rs_batch's closed loop through the ctypes mirror, one run_host call per window with get_state between them
    (as test_ue_rate_hist_gpu's mirror): the twin's [P][S][n_bins]."""
    profs = [sched.load_slice_config(c) for c in cfgs]
    tr = [sched.load_traffic_config(t, c) for c, t in zip(cfgs, trafs)]
    P, nb = len(profs), tr[0][0]
    w, p, u2s = profs[0]
    S, U = len(w), len(u2s)
    cp = np.arange(B) % P
    if P == 1:
        g = sched.Scheduler(algo, w, p, u2s, B, cqi_per_rb=2, n_bearers=nb)
    else:
        g = sched.Scheduler.from_profiles(algo, profs, cp.astype(np.int32), cqi_per_rb=2, n_bearers=nb)
    g.enable_buffers(rbb.K, np.stack([tr[k][1] for k in cp]))
    all_u2s = np.stack([pr[2] for pr in profs])
    arr = workload.synth_arrivals(seed, 0, B, 0, T, all_u2s, np.stack([t[2] for t in tr]), np.stack([t[3] for t in tr]),
                                  n_bearers=nb, cell_profile=cp)
    now, dts = workload.tti_clock(T)
    draws = workload.synth_rand2(seed, 0, B, 0, T, S)
    cqi = sched.pack_cqi(workload.synth_cqi(seed, 0, B, 0, T, U, rbb.G))
    want = np.zeros((P, S, n_bins), np.uint64)
    prev = _cum(g)
    for t0 in range(0, T, W):
        sl = slice(t0, t0 + W)
        res = g.run_host(cqi[sl], draws[sl], dts[sl], ttis_per_launch=16, arrivals=arr[sl], now=now[sl])
        cur = _cum(g)
        want += workload.ue_upt_hist(res["queue_out"], prev, cur, all_u2s, S, n_bins, upt_bytes, cp)
        prev = cur
    g.close()
    return want


@pytest.mark.parametrize("nb,P", [(1, 1), (2, 2)])
def test_rs_batch_equals_python_mirror(nb, P, tmp_path):
    B, T, seed, W, n_bins, rate_bytes, upt_bytes = 19, 45, 6, 9, 30, 6000, 500
    cfgs, trafs = zip(*[rbb._files(tmp_path, nb, tag=str(p), traffic=rbb.TRAFFIC if p == 0 else rbb.TRAFFIC[::-1])
                        for p in range(P)])
    args = ["--algo", 9, "--cells", B, "--ttis", T, "--seed", seed, "--buffers", rbb.K,
            "--rate-window", W, "--rate-bins", n_bins, "--rate-bin-bytes", rate_bytes]
    for c, t in zip(cfgs, trafs):
        args += ["--config", c, "--traffic", t]
    plain = rbb._run(*args)
    lines = rbb._run(*args, "--upt-bin-bytes", upt_bytes)
    hist = _batch_mirror(9, cfgs, trafs, B, T, seed, W, n_bins, upt_bytes)
    assert len(lines) == P
    keys = ["upt_samples", "upt_p5", "upt_p50", "upt_p95"]
    for p, (got, was) in enumerate(zip(lines, plain)):
        assert {k: v for k, v in got.items() if k not in keys and k != "cell_ttis_per_s"} == \
               {k: v for k, v in was.items() if k != "cell_ttis_per_s"}
        assert list(got)[-4:] == keys
        h = hist[p]
        assert got["upt_samples"] == [int(x) for x in h.sum(axis=1)]
        for q in (5, 50, 95):
            assert got[f"upt_p{q}"] == [sched.hist_percentile(h[s], q) for s in range(h.shape[0])], q
    assert hist.sum() > 0 and np.count_nonzero(hist.sum(axis=(0, 1))) >= 3


def test_rs_batch_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 --upt-bin-bytes is compared with --gpus 1 only where two are present")
    cfg, traffic = rbb._files(tmp_path, 2)
    runs = [rbb._run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", rbb.K, "--cells", 301, "--ttis", 64,
                     "--seed", 3, "--gpus", n, "--rate-window", 16, "--rate-bins", 50, "--rate-bin-bytes", 3000,
                     "--upt-bin-bytes", 400)[0] for n in (1, 2)]
    keys = [k for k in runs[0] if k.startswith("upt_")]
    assert len(keys) == 4 and all(runs[0][k] == runs[1][k] for k in keys)
    assert sum(runs[0]["upt_samples"]) > 0

"""GPU: per-UE throughput histograms over caller-closed windows (rs_enable_ue_rate_hist / rs_close_ue_rate_window /
rs_get_ue_rate_hist / rs_ue_rate_hist_device / rs_reduce_ue_rate_hist, rs_batch --rate-window), tolerance 0: the device
counts equal workload.ue_rate_hist fed the cum_bytes get_state returns between the same windows, for every id, every
run entry point, split batches, two bearers, profiles, buffered handles and state changes."""
import ctypes as C

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import SRC_NONE, SRC_ONOFF, SRC_PERIODIC, SRC_RATE
from tests import test_rs_batch_buffers_gpu as rbb
from tests.test_buffers_gpu import K, Traffic
from tests.test_channel_gpu import COUNTS, EDGE_SPEC, SPEC, _channel_cqi, _channel_file
from tests.test_host_api_gpu import _nccl
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu
BINS, BIN_BYTES = 40, 4000


def _torch(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _window(c, g, entry, t0, t1, tpl=16, close=True):
    """TTIs [t0, t1) of Case c through one entry point (rs_step: one call per TTI), then the window's close; the async
    entry points close it before rs_wait, the device ones before the synchronisation."""
    L, B, U, n = sched.lib(), c.B, c.U, t1 - t0
    sl = slice(t0, t1)
    act = None if c.active is None else np.ascontiguousarray(c.active[sl])
    q = None if c.queue is None else c.queue[sl]
    h = None if c.hol is None else c.hol[sl]
    if entry == "step":
        for t in range(t0, t1):
            g.step(c.slabs[t], c.draws[t], dt=float(c.dts[t]), active=None if act is None else act[t - t0],
                   queue=None if q is None else q[t - t0], hol=None if h is None else h[t - t0])
    elif entry == "run_host":
        g.run_host(c.slabs[sl], c.draws[sl], c.dts[sl], active=act, ttis_per_launch=tpl, queue=q, hol=h)
    elif entry == "run_traces_host":
        g.run_traces_host(c.rows[sl], c.draws[sl], c.dts[sl], active=act, ttis_per_launch=tpl, queue=q, hol=h)
    elif entry in ("run_host_async", "run_traces_host_async"):
        out, o = g._host_outputs(n, False)
        keep = g._queues(q, h, (n, B))
        draws, dt = g._draws(c.draws[sl], (n, B)), np.ascontiguousarray(c.dts[sl])
        ticket = C.c_int64(-1)
        if entry == "run_host_async":
            cqi = np.ascontiguousarray(c.slabs[sl])
            rc = L.rs_run_host_async(g._h, n, sched._ptr(cqi), 1, sched._ptr(draws), sched._ptr(act), sched._ptr(dt),
                                     C.byref(o), tpl, C.byref(ticket))
        else:
            rows = np.ascontiguousarray(c.rows[sl])
            rc = L.rs_run_traces_host_async(g._h, n, sched._ptr(rows), sched._ptr(draws), sched._ptr(act),
                                            sched._ptr(dt), C.byref(o), tpl, C.byref(ticket))
        sched._check(rc)
        if close:
            g.close_ue_rate_window()   # the call's kernels may still run: the close is ordered after them
        g.wait(ticket.value)
        del keep, out
        return
    else:
        d_draws = _torch(c.draws[sl]) if g.rand_stride else None
        d_act = None if act is None else _torch(act)
        d_q, d_h = (None, None) if q is None else (_torch(q), _torch(h))
        kw = dict(d_active=0 if d_act is None else d_act.data_ptr(), active_tti_stride=B * U, ttis_per_launch=tpl,
                  d_queue=0 if d_q is None else d_q.data_ptr(), d_hol=0 if d_h is None else d_h.data_ptr())
        r2 = 0 if d_draws is None else d_draws.data_ptr()
        if entry == "run_device":
            d_cqi = _torch(c.slabs[sl])
            g.run_device(n, d_cqi.data_ptr(), d_cqi[0].numel(), r2, c.dts[sl], **kw)
        else:
            g.run_traces_device(n, c.rows[sl], r2, c.dts[sl], **kw)
        if close:
            g.close_ue_rate_window()
        g.sync()
        return
    if close:
        g.close_ue_rate_window()


def _cum(g):
    return g.get_state()["cum_bytes"]


def _check_windows(c, g, windows, u2s, cp=None, bins=BINS, bin_bytes=BIN_BYTES, entry="run_device", tpl=16):
    """Run the windows [(t0, t1), ...] and return (device counts, twin); the twin sums ue_rate_hist over windows."""
    want = np.zeros((u2s.shape[0], c.S, bins), np.uint64)
    prev = _cum(g)
    for t0, t1 in windows:
        _window(c, g, entry, t0, t1, tpl)
        cur = _cum(g)
        want += workload.ue_rate_hist(prev, cur, u2s, c.S, bins, bin_bytes, cp)
        prev = cur
    return g.get_ue_rate_hist(), want


def _spread(want):
    """Samples in bin 0 (idle UEs) and in at least two other bins."""
    per_bin = want.sum(axis=(0, 1))
    return per_bin[0] > 0 and np.count_nonzero(per_bin[1:]) >= 2


def _windows(T, n):
    edges = np.linspace(0, T, n + 1).astype(int)
    return [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:])]


@pytest.mark.parametrize("algo", IDS)
def test_every_id_equals_twin(algo):
    c = Case(algo, CELLS["narrow"], B=9, T=30, seed=9100 + algo, nb=1 if algo == 1 else 2)
    g = c.scheduler()
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    got, want = _check_windows(c, g, _windows(c.T, 3), c.u2s[None])
    g.close()
    assert got.shape == (1, c.S, BINS) and np.array_equal(got, want)
    assert want.sum() == 3 * c.B * c.U and _spread(want)


ENTRIES = ["step", "run_host", "run_host_async", "run_traces_host", "run_traces_host_async", "run_device",
           "run_traces_device"]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("nb", [1, 2])
def test_every_entry_point_equals_twin(entry, nb):
    trace = "traces" in entry
    c = Case(9 if nb == 2 else 8, CELLS["narrow"], B=7, T=24 if entry == "step" else 40, seed=9200 + nb, trace=trace, nb=nb)
    g = c.scheduler()
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    got, want = _check_windows(c, g, _windows(c.T, 4), c.u2s[None], entry=entry)
    g.close()
    assert np.array_equal(got, want), entry
    assert want.sum() == 4 * c.B * c.U and _spread(want)


@pytest.mark.parametrize("entry", ["run_device", "run_host"])
def test_batch_split_over_streams(entry):
    """2400 narrow cells: the handle runs its batch as two parts on two streams; the close follows their join."""
    c = Case(9, CELLS["narrow"], B=2400, T=40, seed=9300, nb=2, active=False)
    g = c.scheduler()
    g.enable_ue_rate_hist(1000, 50)   # bins past the 64 counted in shared memory, and the last bin
    got, want = _check_windows(c, g, _windows(c.T, 2), c.u2s[None], bins=1000, bin_bytes=50, entry=entry, tpl=8)
    g.close()
    assert np.array_equal(got, want)
    assert want[..., 1:64].sum() > 0 and want[..., 64:-1].sum() > 0 and want[..., -1].sum() > 0


def test_three_profiles_moved_between_windows():
    """rs_set_cell_profiles between windows: the later samples go to each cell's new profile and its slices."""
    c = Case(9, CELLS["narrow"], B=12, T=45, seed=9400, nb=2)
    u2s = np.stack([np.roll(c.u2s, 3 * p) for p in range(3)])
    cp = np.arange(c.B) % 3
    g = sched.Scheduler.from_profiles(c.algo, [(c.w, c.p, m) for m in u2s], cp.astype(np.int32), **c.cfg())
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    want = np.zeros((3, c.S, BINS), np.uint64)
    prev = _cum(g)
    for k, (t0, t1) in enumerate(_windows(c.T, 3)):
        if k:
            cp = (cp + 1 + k) % 3
            g.set_cell_profiles(cp.astype(np.int32))
        _window(c, g, "run_host", t0, t1)
        cur = _cum(g)
        want += workload.ue_rate_hist(prev, cur, u2s, c.S, BINS, BIN_BYTES, cp)
        prev = cur
    got = g.get_ue_rate_hist()
    g.close()
    assert got.shape == (3, c.S, BINS) and np.array_equal(got, want)
    assert all(want[p].sum() > 0 for p in range(3)) and _spread(want)


def test_buffered_handle_with_device_sources_and_channel():
    """A buffered handle fed by rs_synth_traffic (RATE, PERIODIC, ONOFF and backlogged slices) and rs_synth_channel
    (fading and i.i.d. slices); the HoL histogram on as well."""
    import torch
    c = Case(9, CELLS["narrow"], B=11, T=60, seed=9500, nb=2, active=False)
    on, off = sched.onoff_spec(5, 8)
    kinds = [{"kind": SRC_NONE}, {"kind": SRC_PERIODIC, "period_ttis": 5, "frame_bytes": [20000, 3000, 7000]},
             {"kind": SRC_ONOFF, "pkt_bytes": 900, "period_ttis": 2, "leave_on_q32": on, "leave_off_q32": off},
             {"kind": SRC_RATE, "pkt_bytes": 1500, "pkts_q16": sched.arrival_spec(1500, 4.0)[1]}]
    tr = Traffic(c, seed=1)
    tr.backlogged[:] = (c.u2s % 4 == 0)[None, :, None]
    g = c.scheduler()
    g.enable_buffers(K, tr.backlogged)
    g.enable_hol_hist(24)
    g.set_sources([kinds[s % 4] for s in range(c.S)])
    g.set_channels([sched.channel_spec(COUNTS, 1.5, 6, 4) if s % 2 else {"kind": workload.CH_IID} for s in range(c.S)])
    g.enable_ue_rate_hist(BINS, 2000)
    per = (c.T, c.B, c.U, 2)
    d_arr = torch.zeros(per, dtype=torch.int32, device="cuda")
    d_cqi = torch.zeros((c.T, c.B, c.U, c.G), dtype=torch.uint8, device="cuda")
    g.synth_traffic(5, 0, 0, c.T, d_arr.data_ptr())
    g.synth_channel(5, 0, 0, c.T, d_cqi.data_ptr())
    d_draws = _torch(c.draws)
    want = np.zeros((1, c.S, BINS), np.uint64)
    prev = _cum(g)
    for t0, t1 in _windows(c.T, 3):
        g.run_device(t1 - t0, d_cqi[t0].data_ptr(), d_cqi[0].numel(), d_draws[t0].data_ptr(), c.dts[t0:t1],
                     ttis_per_launch=16, d_arrivals=d_arr[t0].data_ptr(), now=c.now[t0:t1], arrival_time=tr.at[t0:t1])
        g.close_ue_rate_window()
        cur = _cum(g)
        want += workload.ue_rate_hist(prev, cur, c.u2s, c.S, BINS, 2000)
        prev = cur
    got = g.get_ue_rate_hist()
    assert g.get_hol_hist().sum() > 0
    g.close()
    assert np.array_equal(got, want) and _spread(want)


@pytest.mark.parametrize("nb", [1, 2])
def test_state_changes_restart_the_window(nb):
    """rs_set_state with counters just below 2^32 and near 2^64 (a window that wraps), rs_reset_state mid-run: the
    restarted window matches the twin from the new counters, whatever the window ran before the change."""
    c = Case(9 if nb == 2 else 10, CELLS["narrow"], B=8, T=50, seed=9600 + nb, nb=nb)
    g = c.scheduler()
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    rng = np.random.default_rng(nb)
    shape = (c.B, c.U) if nb == 1 else (c.B, c.U, 2)
    want = np.zeros((1, c.S, BINS), np.uint64)
    prev = _cum(g)
    for k, (t0, t1) in enumerate(_windows(c.T, 5)):
        if k in (1, 3):   # mid-window: the TTIs of the window so far are dropped with the old counters
            _window(c, g, "run_device", t0, t0 + 3, close=False)
            t0 += 3
            base = (1 << 32) - 20000 if k == 1 else (1 << 64) - 20000
            prev = (np.uint64(base) + rng.integers(0, 15000, shape).astype(np.uint64)).astype(np.uint64)
            g.set_state(cum_bytes=prev)
        if k == 4:
            _window(c, g, "run_host", t0, t0 + 2, close=False)
            t0 += 2
            g.reset_state()
            prev = np.zeros(shape, np.uint64)
        _window(c, g, "run_device" if k % 2 else "run_host", t0, t1)
        cur = _cum(g)
        if k == 3:
            assert (cur < prev).any()   # some counters wrapped past 2^64 in this window
        want += workload.ue_rate_hist(prev, cur, c.u2s, c.S, BINS, BIN_BYTES)
        prev = cur
    got = g.get_ue_rate_hist()
    g.close()
    assert np.array_equal(got, want) and want.sum() == 5 * c.B * c.U and _spread(want)


def test_back_to_back_closes():
    """Two closes with no TTI between them: a bin-0 sample per UE; a close right after enabling as well."""
    c = Case(8, CELLS["narrow"], B=5, T=20, seed=9700)
    g = c.scheduler()
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    g.close_ue_rate_window()
    assert g.get_ue_rate_hist()[0, :, 0].sum() == c.B * c.U and g.get_ue_rate_hist().sum() == c.B * c.U
    got, want = _check_windows(c, g, [(0, 20)], c.u2s[None])
    g.close_ue_rate_window()
    g.close_ue_rate_window()
    want[0, :, 0] += np.bincount(c.u2s, minlength=c.S).astype(np.uint64) * np.uint64(3 * c.B)
    assert np.array_equal(g.get_ue_rate_hist(), want) and want[..., 1:].sum() > 0
    g.close()


def test_schedules_state_buffers_and_hol_do_not_change():
    """A split buffered batch through rs_run_device and a host run: every output, the state, the buffers and the HoL
    counts are the same bits with the throughput histogram on (and windows closed) and off."""
    from tests.test_hol_hist_gpu import _handle, _run
    for entry, B, T in (("run_device", 2400, 20), ("run_host", 7, 33)):
        c = Case(10, CELLS["narrow"], B=B, T=T, seed=9750, nb=2, active=False)
        tr = Traffic(c, seed=3)
        runs = []
        for on in (True, False):
            g, _, _ = _handle(c, tr, 1)
            if on:
                g.enable_ue_rate_hist(BINS, BIN_BYTES)
            res = _run(c, g, tr, entry, 16, True)
            if on:
                g.close_ue_rate_window()
                assert g.get_ue_rate_hist().sum() == c.B * c.U
            runs.append((res, g.get_state(), g.get_buffers(), g.get_stats(), g.get_buffer_stats(), g.get_hol_hist()))
            g.close()
        (r0, s0, b0, t0, f0, h0), (r1, s1, b1, t1, f1, h1) = runs
        for x, y in zip(r0, r1):
            assert np.array_equal(x, y), entry
        for d0, d1 in ((s0, s1), (b0, b1)):
            for k in d0:
                assert np.array_equal(d0[k], d1[k]), (entry, k)
        assert np.array_equal(t0, t1) and np.array_equal(f0, f1) and np.array_equal(h0, h1)


def test_device_copy_zeroing_and_refusals():
    import torch
    c = Case(9, CELLS["narrow"], B=5, T=30, seed=9800)
    g = c.scheduler()
    for call in (g.get_ue_rate_hist, g.close_ue_rate_window):
        with pytest.raises(sched.RsError, match="no throughput histogram"):
            call()
    assert sched.lib().rs_ue_rate_hist_bins(g._h) == 0
    for n, x, what in [(-1, 100, "n_bins -1 outside 0..65536"), (65537, 100, "n_bins 65537"),
                       (4, 0, "bin_bytes 0 is not >= 1"), (4, -7, "bin_bytes -7")]:
        with pytest.raises(sched.RsError, match=what):
            g.enable_ue_rate_hist(n, x)
    S = 64   # 65 profiles x 64 slices x 65536 bins of uint64: 2080 MiB
    u2s = np.repeat(np.arange(S), 2).astype(np.int32)
    big = sched.Scheduler.from_profiles(9, [(np.full(S, 1 / S), np.tile(c.p[:1], (S, 1)), u2s)] * 65,
                                        np.arange(65, dtype=np.int32))
    with pytest.raises(sched.RsError, match="exceed 2 GiB"):
        big.enable_ue_rate_hist(65536, 1)
    big.enable_ue_rate_hist(16384, 1)
    big.close()
    g.enable_ue_rate_hist(3, 1)   # every UE with 2 bytes or more in the last bin
    got, want = _check_windows(c, g, [(0, 30)], c.u2s[None], bins=3, bin_bytes=1)
    assert np.array_equal(got, want) and got[0, :, 2].sum() > 0
    d = torch.full((c.S * 3,), 7, dtype=torch.int64, device="cuda")
    g.ue_rate_hist_device(d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64).reshape(got.shape), got)
    g.enable_ue_rate_hist(10, 250)   # again: zeroed, and the window starts from the counters now
    assert sched.lib().rs_ue_rate_hist_bins(g._h) == 10 and not g.get_ue_rate_hist().any()
    g.close_ue_rate_window()
    assert g.get_ue_rate_hist()[0, :, 0].sum() == c.B * c.U
    g.enable_ue_rate_hist(0, 0)   # off
    with pytest.raises(sched.RsError, match="rs_get_ue_rate_hist: the handle has no throughput histogram"):
        g.get_ue_rate_hist()
    g.close()


def test_single_rank_reduce_equals_get():
    c = Case(9, CELLS["narrow"], B=6, T=40, seed=9900, nb=2)
    cp = np.arange(c.B) % 2
    g = sched.Scheduler.from_profiles(c.algo, [(c.w, c.p, c.u2s), (c.w, c.p, np.roll(c.u2s, 2))], cp.astype(np.int32),
                                      **c.cfg())
    g.enable_ue_rate_hist(BINS, BIN_BYTES)
    for t0, t1 in _windows(c.T, 2):
        _window(c, g, "run_device", t0, t1)
    L = _nccl()
    L.rs_reduce_ue_rate_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    uid = (C.c_uint8 * 128)()
    assert L.rs_comm_unique_id(uid) == 0, L.rs_nccl_last_error()
    comm = C.c_void_p()
    assert L.rs_comm_init_rank(1, 0, uid, 0, C.byref(comm)) == 0, L.rs_nccl_last_error()
    red = np.zeros((2, c.S, BINS), dtype=np.uint64)
    assert L.rs_reduce_ue_rate_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, L.rs_nccl_last_error()
    assert np.array_equal(red, g.get_ue_rate_hist()) and red.sum() == 2 * c.B * c.U
    g.enable_ue_rate_hist(0, 0)
    assert L.rs_reduce_ue_rate_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) != 0
    assert b"rs_ue_rate_hist_device" in L.rs_nccl_last_error()
    L.rs_comm_destroy(comm)
    g.close()


# ---- rs_batch --rate-window --------------------------------------------------------------------------------------------
def _batch_mirror(algo, cfgs, trafs, chans, B, T, seed, W, n_bins, bin_bytes):
    """rs_batch through the ctypes mirror, one run_host call per window with get_state between them: the twin's
    [P][S][n_bins].  trafs None: backlogged (no --buffers); chans: the channel files (--channel) or None."""
    profs = [sched.load_slice_config(c) for c in cfgs]
    P = len(profs)
    w, p, u2s = profs[0]
    S, U = len(w), len(u2s)
    cp = np.arange(B) % P
    all_u2s = np.stack([pr[2] for pr in profs])
    nb = 1 if trafs is None else sched.load_traffic_config(trafs[0], cfgs[0])[0]
    if P == 1:
        g = sched.Scheduler(algo, w, p, u2s, B, cqi_per_rb=2, n_bearers=nb)
    else:
        g = sched.Scheduler.from_profiles(algo, profs, cp.astype(np.int32), cqi_per_rb=2, n_bearers=nb)
    now, dts = workload.tti_clock(T)
    draws = workload.synth_rand2(seed, 0, B, 0, T, S)
    cqi = workload.synth_cqi(seed, 0, B, 0, T, U, rbb.G) if chans is None else _channel_cqi(cfgs, chans, B, T, seed)
    cqi = sched.pack_cqi(cqi)
    arr = None
    if trafs is not None:
        tr = [sched.load_traffic_config(t, c) for c, t in zip(cfgs, trafs)]
        g.enable_buffers(rbb.K, np.stack([tr[k][1] for k in cp]))
        arr = workload.synth_arrivals(seed, 0, B, 0, T, all_u2s, np.stack([t[2] for t in tr]),
                                      np.stack([t[3] for t in tr]), n_bearers=nb, cell_profile=cp)
    want = np.zeros((P, S, n_bins), np.uint64)
    prev = _cum(g)
    for t0 in range(0, T, W):
        sl = slice(t0, t0 + W)
        kw = {} if arr is None else dict(arrivals=arr[sl], now=now[sl])
        g.run_host(cqi[sl], draws[sl], dts[sl], ttis_per_launch=16, **kw)
        cur = _cum(g)
        want += workload.ue_rate_hist(prev, cur, all_u2s, S, n_bins, bin_bytes, cp)
        prev = cur
    g.close()
    return want


@pytest.mark.parametrize("kind,P", [("backlogged", 1), ("backlogged", 2), ("closed_loop_channel", 2)])
def test_rs_batch_equals_python_mirror(kind, P, tmp_path):
    B, T, seed, W, n_bins, bin_bytes = 19, 45, 6, 9, 30, 6000
    closed = kind != "backlogged"
    cfgs, trafs = zip(*[rbb._files(tmp_path, 2 if closed else 1, tag=str(p),
                                   groups=rbb.GROUPS if p == 0 else [(n, w, (a, b, 1 - e, s)) for n, w, (a, b, e, s) in rbb.GROUPS[::-1]],
                                   traffic=rbb.TRAFFIC if p == 0 else rbb.TRAFFIC[::-1]) for p in range(P)])
    chans = None
    args = ["--algo", 9, "--cells", B, "--ttis", T, "--seed", seed]
    if closed:
        chans = [_channel_file(tmp_path, [SPEC, EDGE_SPEC, {"iid": 1}], 7, tag=str(p)) for p in range(P)]
        args += ["--buffers", rbb.K]
        for c, t, h in zip(cfgs, trafs, chans):
            args += ["--config", c, "--traffic", t, "--channel", h]
    else:
        for c in cfgs:
            args += ["--config", c]
    plain = rbb._run(*args)
    lines = rbb._run(*args, "--rate-window", W, "--rate-bins", n_bins, "--rate-bin-bytes", bin_bytes)
    hist = _batch_mirror(9, cfgs, trafs if closed else None, chans, B, T, seed, W, n_bins, bin_bytes)
    assert len(lines) == P
    keys = ["ue_rate_samples", "ue_rate_p5", "ue_rate_p50", "ue_rate_p95"]
    for p, (got, was) in enumerate(zip(lines, plain)):
        assert {k: v for k, v in got.items() if k not in keys and k != "cell_ttis_per_s"} == \
               {k: v for k, v in was.items() if k != "cell_ttis_per_s"}
        assert list(got)[-4:] == keys
        h = hist[p]
        assert got["ue_rate_samples"] == [int(x) for x in h.sum(axis=1)]
        for q in (5, 50, 95):
            assert got[f"ue_rate_p{q}"] == [sched.hist_percentile(h[s], q) for s in range(h.shape[0])], q
    assert hist.sum() == (T // W) * B * sum(rbb.UES)
    assert np.count_nonzero(hist.sum(axis=(0, 1))) >= 3


def test_rs_batch_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 --rate-window is compared with --gpus 1 only where two are present")
    cfg, traffic = rbb._files(tmp_path, 2)
    runs = [rbb._run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", rbb.K, "--cells", 301, "--ttis", 64,
                     "--seed", 3, "--gpus", n, "--rate-window", 16, "--rate-bins", 50, "--rate-bin-bytes", 3000)[0]
            for n in (1, 2)]
    keys = [k for k in runs[0] if k.startswith("ue_rate_")]
    assert len(keys) == 4 and all(runs[0][k] == runs[1][k] for k in keys)
    assert sum(runs[0]["ue_rate_samples"]) == 4 * 301 * sum(rbb.UES)

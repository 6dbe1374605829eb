"""GPU: head-of-line delay histograms of buffered handles (rs_enable_hol_hist / rs_get_hol_hist / rs_hol_hist_device /
rs_reduce_hol_hist, rs_batch --hol-bins), tolerance 0: the device counts equal workload.hol_hist computed from the same
run's queue_out / hol_out / tbs_bits, for every id and every run entry point, and row 0 equals the hol_delay fields of
the reference's stderr lines (rs_log) for the same cells."""
import ctypes as C
import re

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import SRC_NONE, SRC_ONOFF, SRC_PERIODIC, SRC_RATE
from tests import test_rs_batch_buffers_gpu as rbb
from tests.test_buffers_gpu import K, Traffic
from tests.test_host_api_gpu import _nccl
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu
BINS = 24   # 1-TTI bins


def _torch(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _handle(c, tr, P, bins=BINS, per_unit=1000.0):
    """A buffered handle of Case c (P profiles: rolled slice maps, cell b on profile b % P) with the histogram on;
    returns (handle, u2s [P][U], cell_profile)."""
    if P == 1:
        g, u2s, cp = c.scheduler(), c.u2s[None], None
    else:
        u2s = np.stack([np.roll(c.u2s, 3 * p) for p in range(P)])
        cp = np.arange(c.B) % P
        g = sched.Scheduler.from_profiles(c.algo, [(c.w, c.p, m) for m in u2s], cp.astype(np.int32), **c.cfg())
        if c.trace:
            g.set_traces(c.traces, c.ue_trace)
    g.enable_buffers(K, tr.backlogged)
    if bins:
        g.enable_hol_hist(bins, per_unit)
    return g, u2s, cp


def _twin(c, tr, u2s, cp, q, h, tbs, bins=BINS, per_unit=1000.0):
    return workload.hol_hist(q, h, tbs, c.algo, u2s, tr.backlogged, c.S, bins, per_unit, cp)


def _host_run(c, g, tr, entry, tpl, want_tbs):
    """One call of a host entry point over the whole run (rs_step: one call per TTI); returns (queue, hol, tbs or None).
    want_tbs False: the handle's own scratch feeds the histogram."""
    L, T, B = sched.lib(), c.T, c.B
    outs = []
    for t0, n in ([(t, 1) for t in range(T)] if entry == "step" else [(0, T)]):
        lead = None if entry == "step" else n
        out, o = g._host_outputs(lead, False)
        if not want_tbs:
            o.tbs_bits = None
        sl = slice(t0, t0 + n)
        arr = tr.arr[t0] if entry == "step" else tr.arr[sl]
        keep = g._traffic(arr, c.now[sl], tr.at[sl], lead, out)
        draws = np.ascontiguousarray(c.draws[t0] if entry == "step" else c.draws[sl])
        dt = np.ascontiguousarray(c.dts[sl])
        ticket = C.c_int64(-1)
        if entry == "step":
            rc = L.rs_step(g._h, sched._ptr(np.ascontiguousarray(c.slabs[t0])), sched._ptr(draws), None, float(dt[0]),
                           C.byref(o))
        elif entry in ("run_host", "run_host_async"):
            args = [g._h, n, sched._ptr(np.ascontiguousarray(c.slabs[sl])), 1, sched._ptr(draws), None, sched._ptr(dt),
                    C.byref(o), tpl]
            rc = L.rs_run_host(*args) if entry == "run_host" else L.rs_run_host_async(*args, C.byref(ticket))
        else:
            args = [g._h, n, sched._ptr(np.ascontiguousarray(c.rows[sl])), sched._ptr(draws), None, sched._ptr(dt),
                    C.byref(o), tpl]
            rc = L.rs_run_traces_host(*args) if entry == "run_traces_host" else L.rs_run_traces_host_async(*args, C.byref(ticket))
        sched._check(rc)
        if ticket.value >= 0:
            g.wait(ticket.value)
        del keep
        outs.append((out["queue_out"].reshape((n, B) + out["queue_out"].shape[-2 if c.nb == 2 else -1:]),
                     out["hol_out"].reshape((n, B) + out["hol_out"].shape[-2 if c.nb == 2 else -1:]),
                     out["tbs_bits"].reshape(n, B, c.U)))
    q, h, tbs = (np.concatenate(x) for x in zip(*outs))
    return q, h, tbs if want_tbs else None


def _device_run(c, g, tr, entry, tpl, want_out):
    """rs_run_device / rs_run_traces_device over the whole run; want_out False: no queue_out / hol_out / tbs_bits (the
    handle's scratch).  Returns (queue, hol, tbs) or None."""
    import torch
    T, B, U = c.T, c.B, c.U
    per = tr.arr.shape
    d_arr, d_draws = _torch(tr.arr), _torch(c.draws)
    d_q = torch.zeros(per, dtype=torch.int32, device="cuda") if want_out else None
    d_h = torch.zeros(per, dtype=torch.float64, device="cuda") if want_out else None
    d_tbs = torch.zeros((T, B, U), dtype=torch.int32, device="cuda") if want_out else None
    kw = dict(d_out={"tbs_bits": d_tbs.data_ptr()} if want_out else None, ttis_per_launch=tpl, d_arrivals=d_arr.data_ptr(),
              now=c.now, arrival_time=tr.at, d_queue_out=d_q.data_ptr() if want_out else 0,
              d_hol_out=d_h.data_ptr() if want_out else 0)
    if entry == "run_device":
        d_cqi = _torch(c.slabs)
        g.run_device(T, d_cqi.data_ptr(), B * U * c.G, d_draws.data_ptr(), c.dts, **kw)
    else:
        g.run_traces_device(T, c.rows, d_draws.data_ptr(), c.dts, **kw)
    g.sync()
    return (d_q.cpu().numpy(), d_h.cpu().numpy(), d_tbs.cpu().numpy()) if want_out else None


def _run(c, g, tr, entry, tpl, with_out):
    if entry in ("run_device", "run_traces_device"):
        return _device_run(c, g, tr, entry, tpl, with_out)
    q, h, tbs = _host_run(c, g, tr, entry, tpl, with_out)
    return (q, h, tbs) if with_out else None


def _check_entry(algo, nb, P, entry, tpl, T=40, B=9, bins=BINS, per_unit=1000.0, ups=CELLS["narrow"]):
    """The same run with and without the caller's output arrays: both counts equal the twin of the first run's outputs."""
    trace = entry in ("run_traces_host", "run_traces_host_async", "run_traces_device")
    c = Case(algo, ups, B=B, T=T, seed=9700 + algo + 10 * nb + P, trace=trace, nb=nb, active=False)
    tr = Traffic(c, seed=algo + nb + P)
    hists = []
    for with_out in (True, False):
        g, u2s, cp = _handle(c, tr, P, bins, per_unit)
        res = _run(c, g, tr, entry, tpl, with_out)
        if with_out:
            want = _twin(c, tr, u2s, cp, *res, bins=bins, per_unit=per_unit)
        hists.append(g.get_hol_hist())
        g.close()
    assert hists[0].shape == (P, 2, c.S, bins)
    assert np.array_equal(hists[0], want), entry
    assert np.array_equal(hists[1], want), entry + " (scratch)"
    assert want[:, 0, :, 1:].sum() > 0 and want[:, 1, :, 1:].sum() > 0   # delays served and waiting
    return want


@pytest.mark.parametrize("algo", IDS)
def test_every_id_equals_twin(algo):
    _check_entry(algo, 1 if algo == 1 else 2, 1, "run_device", 16)


ENTRIES = ["step", "run_host", "run_host_async", "run_traces_host", "run_traces_host_async", "run_device",
           "run_traces_device"]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("nb,P", [(1, 1), (2, 3)])
def test_every_entry_point_equals_twin(entry, nb, P):
    _check_entry(9 if nb == 2 else 8, nb, P, entry, 16, T=24 if entry == "step" else 40)


@pytest.mark.parametrize("tpl", [1, 16, 64])
@pytest.mark.parametrize("entry", ["run_host", "run_device"])
def test_ttis_per_launch(entry, tpl):
    _check_entry(103, 2, 1, entry, tpl, T=70)


def test_batch_split_over_streams():
    """2400 narrow cells: the handle runs its batch as two parts on two streams, each with its own reducer launches."""
    _check_entry(9, 2, 1, "run_device", 16, T=20, B=2400)
    _check_entry(9, 1, 3, "run_host", 8, T=20, B=2400)


SMEM_BINS = 64   # the reducer counts bins 0..63 in shared memory while 2 x S x P rows of them fit 48 KB (rs_sched.cu)


@pytest.mark.parametrize("entry", ["run_device", "run_host"])
def test_long_delays_on_the_global_path(entry):
    """100 bins per TTI: delays of a few TTIs land on both sides of the shared-memory bins, and past the last bin."""
    want = _check_entry(9, 2, 1, entry, 16, T=40, bins=600, per_unit=1e5)
    assert want[..., :SMEM_BINS].sum() > 0 and want[..., SMEM_BINS:-1].sum() > 0
    assert want[:, 1, :, -1].sum() > 0


def test_no_shared_bins():
    """64 slices x 97 profiles: 2 x 64 x 97 rows of even one 32-bit counter exceed 48 KB, so every sample is added to
    global memory."""
    assert 2 * 64 * 97 * 4 > 48 * 1024
    want = _check_entry(8, 2, 97, "run_device", 16, T=24, B=97, bins=30, ups=[2] * 64)
    assert want[..., 1:].sum() > 0


def test_device_drawn_traffic():
    """Arrivals drawn by rs_synth_traffic from RATE, PERIODIC and ONOFF sources (and a slice without one)."""
    import torch
    c = Case(9, CELLS["narrow"], B=11, T=60, seed=9800, nb=2, active=False)
    on, off = sched.onoff_spec(5, 8)
    kinds = [{"kind": SRC_NONE}, {"kind": SRC_PERIODIC, "period_ttis": 5, "frame_bytes": [20000, 3000, 7000]},
             {"kind": SRC_ONOFF, "pkt_bytes": 900, "period_ttis": 2, "leave_on_q32": on, "leave_off_q32": off},
             {"kind": SRC_RATE, "pkt_bytes": 1500, "pkts_q16": sched.arrival_spec(1500, 4.0)[1]}]
    src = [kinds[s % 4] for s in range(c.S)]
    tr = Traffic(c, seed=1)
    tr.backlogged[:] = (c.u2s % 4 == 0)[None, :, None]
    g, u2s, cp = _handle(c, tr, 1)
    g.set_sources(src)
    per = (c.T, c.B, c.U, 2)
    d_arr = torch.zeros(per, dtype=torch.int32, device="cuda")
    g.synth_traffic(5, 0, 0, c.T, d_arr.data_ptr())
    tr.arr = d_arr.cpu().numpy()
    res = _device_run(c, g, tr, "run_device", 16, True)
    want = _twin(c, tr, u2s, cp, *res)
    assert np.array_equal(g.get_hol_hist(), want)
    assert all(want[0, 1, s].sum() > 0 for s in range(c.S) if s % 4)   # every kind queues
    g.close()


@pytest.mark.parametrize("algo,nb,P", [(9, 1, 1), (7, 2, 3), (1, 1, 1)])
def test_row0_equals_the_reference_stderr_lines(algo, nb, P):
    """Row 0 over a small batch equals the histogram of the hol_delay fields rs_log prints for every cell's FIFO
    bearers (arrival time = now: the delays sit on whole TTIs, far from a bin edge, so %g's digits bin alike)."""
    c = Case(algo, CELLS["narrow"], B=6, T=50, seed=9900 + algo, nb=nb, active=False)
    tr = Traffic(c, seed=algo)
    tr.at = c.now
    g, u2s, cp = _handle(c, tr, P)
    res = g.run_host(c.slabs, c.draws, c.dts, want_aux=True, ttis_per_launch=16, arrivals=tr.arr, now=c.now,
                     arrival_time=c.now)
    hist = g.get_hol_hist()
    g.close()
    want = np.zeros((P, c.S, BINS), np.uint64)
    line = re.compile(r"^\d+ app: (\d+) cumu_bytes: \d+ cumu_rbs: \d+ hol_delay: (\S+) user: (\d+) slice: (\d+)$")
    lines = 0
    for b in range(c.B):
        p = 0 if cp is None else int(cp[b])
        lw = sched.LogWriter(algo, u2s[p], c.S, n_bearers=nb)
        for t in range(c.T):
            transport = algo in (8, 9, 101, 103)
            lw.tti(100 + t, c.slabs[t, b], res["rbg_to_ue"][t, b], res["tbs_bits"][t, b],
                   res["final_cqi"][t, b] if algo != 1 else None, res["slice_target"][t, b] if transport else None,
                   res["slice_quota"][t, b] if transport else None, queue=res["queue_out"][t, b], hol=res["hol_out"][t, b])
        for ln in lw.stderr.splitlines():
            m = line.match(ln)
            if not m:
                continue
            app, hol, u, s = int(m.group(1)), float(m.group(2)), int(m.group(3)), int(m.group(4))
            if tr.backlogged.reshape(c.B, c.U, nb)[b, u, app - u * nb]:
                continue
            want[p, s, min(int(np.floor(hol * 1000.0 + 0.5)), BINS - 1)] += np.uint64(1)
            lines += 1
        lw.close()
    assert lines > c.T and np.array_equal(hist[:, 0], want)


def test_schedules_state_and_buffers_do_not_change():
    """A split batch through rs_run_device and a host run: every output, the state and the buffers are the same bits with
    the histogram on and off."""
    for entry, B, T in (("run_device", 2400, 20), ("run_host", 7, 33)):
        c = Case(10, CELLS["narrow"], B=B, T=T, seed=9950, nb=2, active=False)
        tr = Traffic(c, seed=3)
        runs = []
        for bins in (BINS, 0):
            g, _, _ = _handle(c, tr, 1, bins=bins)
            res = _run(c, g, tr, entry, 16, True)
            runs.append((res, g.get_state(), g.get_buffers(), g.get_stats(), g.get_buffer_stats()))
            g.close()
        (r0, s0, b0, t0, f0), (r1, s1, b1, t1, f1) = runs
        for x, y in zip(r0, r1):
            assert np.array_equal(x, y), entry
        for d0, d1 in ((s0, s1), (b0, b1)):
            for k in d0:
                assert np.array_equal(d0[k], d1[k]), (entry, k)
        assert np.array_equal(t0, t1) and np.array_equal(f0, f1)


def test_device_copy_zeroing_and_refusals():
    import torch
    c = Case(9, CELLS["narrow"], B=5, T=30, seed=9960, active=False)
    tr = Traffic(c, seed=2)
    g = c.scheduler()
    for call in (lambda: g.enable_hol_hist(8), g.get_hol_hist):
        with pytest.raises(sched.RsError, match="no buffers|no delay histogram"):
            call()
    g.enable_buffers(K, tr.backlogged)
    with pytest.raises(sched.RsError, match="rs_get_hol_hist: the handle has no delay histogram"):
        g.get_hol_hist()
    for n, bpu, what in [(-1, 1000.0, "n_bins -1 outside 0..65536"), (65537, 1000.0, "n_bins 65537"),
                         (4, 0.0, "bins_per_unit 0"), (4, float("inf"), "bins_per_unit inf"),
                         (4, float("nan"), "bins_per_unit nan")]:
        with pytest.raises(sched.RsError, match=what):
            g.enable_hol_hist(n, bpu)
    S = 64   # 40 profiles x 2 x 64 slices x 65536 bins of uint64: 2.5 GiB
    u2s = np.repeat(np.arange(S), 2).astype(np.int32)
    big = sched.Scheduler.from_profiles(9, [(np.full(S, 1 / S), np.tile(c.p[:1], (S, 1)), u2s)] * 40,
                                        np.arange(40, dtype=np.int32))
    big.enable_buffers(2)
    with pytest.raises(sched.RsError, match="exceed 2 GiB"):
        big.enable_hol_hist(65536)
    big.enable_hol_hist(16384)
    big.close()
    g.enable_hol_hist(3, 1000.0)   # every delay of 2 TTIs or more in the last bin
    res = _device_run(c, g, tr, "run_device", 16, True)
    got = g.get_hol_hist()
    assert np.array_equal(got, _twin(c, tr, c.u2s[None], None, *res, bins=3)) and got[0, 1, :, 2].sum() > 0
    d = torch.full((2 * c.S * 3,), 7, dtype=torch.int64, device="cuda")
    g.hol_hist_device(d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64).reshape(got.shape), got)
    g.enable_hol_hist(10, 250.0)   # again: zeroed
    assert not g.get_hol_hist().any()
    g.enable_buffers(K, tr.backlogged)   # the buffers again: the histogram is off
    with pytest.raises(sched.RsError, match="no delay histogram"):
        g.get_hol_hist()
    g.close()


def test_single_rank_reduce_equals_get():
    c = Case(9, CELLS["narrow"], B=6, T=40, seed=9970, nb=2, active=False)
    tr = Traffic(c, seed=4, n_profiles=2, cell_profile=np.arange(c.B) % 2)
    g, _, _ = _handle(c, tr, 2)
    _device_run(c, g, tr, "run_device", 16, False)
    L = _nccl()
    L.rs_reduce_hol_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    uid = (C.c_uint8 * 128)()
    assert L.rs_comm_unique_id(uid) == 0, L.rs_nccl_last_error()
    comm = C.c_void_p()
    assert L.rs_comm_init_rank(1, 0, uid, 0, C.byref(comm)) == 0, L.rs_nccl_last_error()
    red = np.zeros((2, 2, c.S, BINS), dtype=np.uint64)
    assert L.rs_reduce_hol_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, L.rs_nccl_last_error()
    assert np.array_equal(red, g.get_hol_hist()) and red.sum() > 0
    g.enable_hol_hist(0)
    assert L.rs_reduce_hol_hist(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) != 0
    assert b"rs_hol_hist_device" in L.rs_nccl_last_error()
    L.rs_comm_destroy(comm)
    g.close()


# ---- rs_batch --hol-bins -----------------------------------------------------------------------------------------------
def _batch_mirror(algo, cfgs, trafs, B, T, seed, n_bins):
    """rs_batch's closed loop through the ctypes mirror (as test_rs_batch_buffers_gpu.mirror): the twin's [P][2][S][n]."""
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
    bl = np.stack([tr[c][1] for c in cp])
    g.enable_buffers(rbb.K, bl)
    all_u2s = np.stack([pr[2] for pr in profs])
    arr = workload.synth_arrivals(seed, 0, B, 0, T, all_u2s, np.stack([t[2] for t in tr]), np.stack([t[3] for t in tr]),
                                  n_bearers=nb, cell_profile=cp)
    now, dts = workload.tti_clock(T)
    draws = workload.synth_rand2(seed, 0, B, 0, T, S)
    res = g.run_host(sched.pack_cqi(workload.synth_cqi(seed, 0, B, 0, T, U, rbb.G)), draws, dts, ttis_per_launch=16,
                     arrivals=arr, now=now)
    g.close()
    return workload.hol_hist(res["queue_out"], res["hol_out"], res["tbs_bits"], algo, all_u2s, bl, S, n_bins, 1000.0, cp)


@pytest.mark.parametrize("nb,P", [(1, 1), (2, 2)])
def test_rs_batch_equals_python_mirror(nb, P, tmp_path):
    B, T, seed, n_bins = 19, 45, 6, 12
    cfgs, trafs = zip(*[rbb._files(tmp_path, nb, tag=str(p), traffic=rbb.TRAFFIC if p == 0 else rbb.TRAFFIC[::-1])
                        for p in range(P)])
    args = ["--algo", 9, "--cells", B, "--ttis", T, "--seed", seed, "--buffers", rbb.K]
    for c, t in zip(cfgs, trafs):
        args += ["--config", c, "--traffic", t]
    plain = rbb._run(*args)
    lines = rbb._run(*args, "--hol-bins", n_bins)
    hist = _batch_mirror(9, cfgs, trafs, B, T, seed, n_bins)
    assert len(lines) == P
    for p, (got, was) in enumerate(zip(lines, plain)):
        extra = {k: v for k, v in got.items() if k.startswith("hol_")}
        assert {k: v for k, v in got.items() if k not in extra and k != "cell_ttis_per_s"} == \
               {k: v for k, v in was.items() if k != "cell_ttis_per_s"}
        assert list(got)[-len(extra):] == list(extra)
        for r, name in enumerate(("hol_served", "hol_waiting")):
            h = hist[p, r]
            assert got[name] == [int(x) for x in h.sum(axis=1)]
            for q in (50, 95, 99):
                assert got[f"{name}_p{q}"] == [sched.hist_percentile(h[s], q) for s in range(h.shape[0])], (name, q)
        assert None in got["hol_served_p50"] and sum(got["hol_waiting"]) > 0   # slice 0 is backlogged: no samples


def test_rs_batch_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 --hol-bins is compared with --gpus 1 only where two are present")
    cfg, traffic = rbb._files(tmp_path, 2)
    runs = [rbb._run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", rbb.K, "--cells", 301, "--ttis", 64,
                     "--seed", 3, "--gpus", n, "--hol-bins", 40)[0] for n in (1, 2)]
    keys = [k for k in runs[0] if k.startswith("hol_")]
    assert len(keys) == 8 and all(runs[0][k] == runs[1][k] for k in keys)

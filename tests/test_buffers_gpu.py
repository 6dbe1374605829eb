"""Per-bearer buffers kept on the device (rs_enable_buffers / rs_set_traffic): the closed loop against the CPU model of
tests/buffer_model.py driving the oracle one TTI at a time, tolerance 0.  Every output of every TTI (including the queue
sizes and delays the TTIs showed), the scheduler state and the buffers at every call boundary are compared.  Each
closed-loop case first asserts that its queues both drain and build up."""
import re

import numpy as np
import pytest

from oracle.pyoracle import OracleScheduler
from radiosaber_b200 import sched, workload
from tests.buffer_model import BufferModel, closed_loop
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

gpu = pytest.mark.gpu
K = 12


class Traffic:
    """Arrivals of a Case from workload.synth_arrivals: per slice a packet size (0 = none) and a rate that either drains
    or overloads the bearers, slice 0 backlogged; arrival times half a TTI before each TTI's `now`."""

    def __init__(self, c, seed, n_profiles=1, cell_profile=None):
        rng = np.random.default_rng(seed)
        S = c.S
        self.pkt = rng.choice([0, 200, 1500], size=(n_profiles, S)).astype(np.int32)
        self.q16 = (rng.choice([0.2, 0.7, 3.5, 9.0], size=(n_profiles, S)) * 65536).astype(np.int32)
        self.pkt[:, 1], self.q16[:, 1] = 1500, 9 * 65536       # always one overloaded slice ...
        self.pkt[:, 2 % S], self.q16[:, 2 % S] = 200, 13107   # ... and one that drains (0.2 packets per TTI)
        self.seed, self.cell_profile = seed, cell_profile
        u2s = c.u2s if n_profiles == 1 else np.stack([c.u2s] * n_profiles)
        self.arr = workload.synth_arrivals(seed, 0, c.B, 0, c.T, u2s, self.pkt, self.q16, n_bearers=c.nb,
                                           cell_profile=cell_profile)
        per = (c.B, c.U) if c.nb == 1 else (c.B, c.U, 2)
        self.backlogged = np.zeros(per, bool)
        self.backlogged[:, c.u2s == 0] = True
        if c.nb == 2:
            self.backlogged[:, c.u2s == 3 % S, 0] = True   # a UE with one backlogged and one buffered bearer
        self.now = c.now
        self.at = c.now - 0.0005

    def model(self, c):
        return BufferModel(self.backlogged.shape, K, self.backlogged)


def oracle_loop(c, tr, bounds):
    o = OracleScheduler(c.algo, c.w, c.p, c.u2s, c.B, cqi_per_rb=1 if c.layout == 1 else 0, n_threads=8,
                        grant_list_len=c.grant_len, **c.cfg())
    return closed_loop(o, tr.model(c), c.ocqi, c.draws, c.dts, tr.arr, tr.now, tr.at, active=c.active, bounds=bounds)


def assert_drains_and_builds(outs, tr):
    q = outs["queue_out"]
    buffered = ~np.broadcast_to(tr.backlogged, q.shape)
    drained = (q[1:] == 0) & (q[:-1] > 0) & buffered[1:]
    assert drained.any(), "no queue ever drained"
    assert q[buffered].max() > 15000, "no queue built up"


def host_run(c, g, tr, bounds, tpl):
    outs, states, bufs, t0 = [], [], [], 0
    for t1 in bounds:
        kw = dict(active=c._sl(c.active, t0, t1), want_aux=True, ttis_per_launch=tpl, arrivals=tr.arr[t0:t1],
                  now=tr.now[t0:t1], arrival_time=tr.at[t0:t1])
        if c.trace:
            outs.append(g.run_traces_host(c.rows[t0:t1], c.draws[t0:t1], c.dts[t0:t1], **kw))
        else:
            outs.append(g.run_host(c.slabs[t0:t1], c.draws[t0:t1], c.dts[t0:t1], **kw))
        states.append(g.get_state())
        bufs.append(g.get_buffers())
        t0 = t1
    return {k: np.concatenate([x[k] for x in outs]) for k in outs[0]}, states, bufs


def device_run(c, g, tr, bounds, tpl):
    import torch
    T, B, U, S, G = c.T, c.B, c.U, c.S, c.G
    per = tr.arr.shape
    out = {"rbg_to_ue": torch.empty((T, B, G), dtype=torch.int16), "tbs_bits": torch.empty((T, B, U), dtype=torch.int32),
           "mcs": torch.empty((T, B, U), dtype=torch.uint8), "final_cqi": torch.empty((T, B, U), dtype=torch.uint8)}
    if c.algo in (8, 9, 10, 101, 103):
        out["slice_target"] = torch.empty((T, B, S), dtype=torch.int32)
        out["slice_quota"] = torch.empty((T, B, S), dtype=torch.int32)
    if c.algo in (7, 11):
        out["nvs_slice"] = torch.empty((T, B), dtype=torch.int32)
    if c.algo == 10:
        out["alloc_n"] = torch.empty((T, B), dtype=torch.int32)
        out["alloc_ue"] = torch.empty((T, B, g.grant_list_len), dtype=torch.int16)
        out["alloc_rbg"] = torch.empty((T, B, g.grant_list_len), dtype=torch.int16)
    out = {k: v.cuda() for k, v in out.items()}
    qo, ho = torch.empty(per, dtype=torch.int32).cuda(), torch.empty(per, dtype=torch.float64).cuda()
    d_arr = torch.empty(per, dtype=torch.int32).cuda()
    g.synth_arrivals(tr.seed, 0, 0, T, tr.pkt, tr.q16, d_arr.data_ptr())   # the device twin feeds the device run
    dev = {k: None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda()
           for k, v in (("draws", c.draws), ("act", c.active))}
    d_slabs = None if c.trace else torch.from_numpy(np.ascontiguousarray(c.slabs)).cuda()
    states, bufs, t0 = [], [], 0
    for t1 in bounds:
        n = t1 - t0
        kw = dict(d_out={k: v[t0].data_ptr() for k, v in out.items()},
                  d_active=0 if dev["act"] is None else dev["act"][t0].data_ptr(), active_tti_stride=B * U,
                  ttis_per_launch=tpl, d_arrivals=d_arr[t0].data_ptr(), now=tr.now[t0:t1], arrival_time=tr.at[t0:t1],
                  d_queue_out=qo[t0].data_ptr(), d_hol_out=ho[t0].data_ptr())
        r2 = dev["draws"][t0].data_ptr() if g.rand_stride else 0
        if c.trace:
            g.run_traces_device(n, c.rows[t0:t1], r2, c.dts[t0:t1], **kw)
        else:
            g.run_device(n, d_slabs[t0].data_ptr(), d_slabs[0].numel(), r2, c.dts[t0:t1], **kw)
        g.sync()
        states.append(g.get_state())
        bufs.append(g.get_buffers())
        t0 = t1
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["queue_out"], res["hol_out"] = qo.cpu().numpy(), ho.cpu().numpy()
    return res, states, bufs


def check(c, got, want, tag=""):
    outs, states, bufs = got
    w_outs, w_states, w_bufs = want
    c.check((outs, states), (w_outs, w_states), tag)
    assert len(bufs) == len(w_bufs)
    for i, (a, b) in enumerate(zip(bufs, w_bufs)):
        for k in b:
            assert np.array_equal(a[k], b[k]), (tag, "buffers", i, k)


def buffered(c, tr, **env):
    g = c.scheduler(**env)
    g.enable_buffers(K, tr.backlogged)
    return g


# ---- 1. oracle parity of the closed loop ---------------------------------------------------------------------------
MATRIX = [(w, a, tr, nb) for w in ("narrow", "wide") for a in IDS for tr in (False, True) for nb in (1, 2)
          if not (a == 1 and nb == 2)]


@gpu
@pytest.mark.parametrize("width,algo,trace,nb", MATRIX)
def test_closed_loop_matches_oracle(width, algo, trace, nb):
    """130 TTIs in two calls, launches of 1, 7 and 64 TTIs, through rs_run_host / rs_run_traces_host."""
    c = Case(algo, CELLS[width], B=4, T=130, seed=7000 + 10 * IDS.index(algo) + 4 * trace + 2 * nb + (width == "wide"),
             trace=trace, nb=nb)
    tr = Traffic(c, seed=algo + 3 * nb + trace)
    bounds = [80, 130]
    want = oracle_loop(c, tr, bounds)
    assert_drains_and_builds(want[0], tr)
    for tpl in (1, 7, 64):
        g = buffered(c, tr)
        check(c, host_run(c, g, tr, bounds, tpl), want, tag=f"ttis_per_launch {tpl}")
        g.close()


# ---- 2. entry points -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("algo,nb", [(1, 1), (7, 2), (9, 1), (9, 2), (10, 2), (11, 1), (103, 2)])
def test_device_entry_points(algo, nb, trace):
    """rs_run_device / rs_run_traces_device with DEVICE arrivals from rs_synth_arrivals and device queue_out / hol_out."""
    c = Case(algo, CELLS["narrow"], B=5, T=70, seed=7500 + algo + nb + trace, trace=trace, nb=nb)
    tr = Traffic(c, seed=31 + algo)
    bounds = [33, 70]
    want = oracle_loop(c, tr, bounds)
    assert_drains_and_builds(want[0], tr)
    g = buffered(c, tr)
    check(c, device_run(c, g, tr, bounds, 7), want, tag="device")
    g.close()


@gpu
@pytest.mark.parametrize("algo,nb", [(9, 1), (7, 2), (1, 1)])
def test_step(algo, nb):
    """rs_step, one TTI per call."""
    c = Case(algo, CELLS["narrow"], B=3, T=40, seed=7600 + algo, nb=nb)
    tr = Traffic(c, seed=algo)
    want = oracle_loop(c, tr, [40])
    assert_drains_and_builds(want[0], tr)
    g = buffered(c, tr)
    outs = []
    for t in range(c.T):
        outs.append(g.step(c.ocqi[t], c.draws[t], dt=float(c.dts[t]), active=c.active[t], want_aux=True,
                           arrivals=tr.arr[t], now=tr.now[t], arrival_time=tr.at[t]))
    got = {k: np.stack([o[k] for o in outs]) for k in outs[0]}
    check(c, (got, [g.get_state()], [g.get_buffers()]), want, tag="rs_step")
    g.close()


@gpu
@pytest.mark.parametrize("env", [{"RS_PARTS": 3}, {"RS_NO_SPLIT": 1}])
@pytest.mark.parametrize("algo,nb", [(9, 2), (10, 1)])
def test_part_batches(algo, nb, env):
    c = Case(algo, CELLS["narrow"], B=7, T=50, seed=7700 + algo + nb, nb=nb)
    tr = Traffic(c, seed=5 + nb)
    bounds = [20, 50]
    want = oracle_loop(c, tr, bounds)
    g = buffered(c, tr, **env)
    check(c, host_run(c, g, tr, bounds, 7), want, tag=f"host {env}")
    g.enable_buffers(K, tr.backlogged)   # enabling again empties the buffers
    g.reset_state()
    check(c, device_run(c, g, tr, bounds, 7), want, tag=f"device {env}")
    g.close()


@gpu
def test_two_async_calls_in_flight():
    """Two rs_run_host_async calls enqueued before the first wait."""
    c = Case(9, CELLS["narrow"], B=4, T=60, seed=7800, nb=2, active=False)
    tr = Traffic(c, seed=77)
    want = oracle_loop(c, tr, [60])
    g = buffered(c, tr)
    keep, tickets, outs = [], [], []
    for t0, t1 in ((0, 30), (30, 60)):
        out, o = g._host_outputs(t1 - t0, True)
        args = (np.ascontiguousarray(c.slabs[t0:t1]), np.ascontiguousarray(c.draws[t0:t1]), np.ascontiguousarray(c.dts[t0:t1]))
        traffic = (np.ascontiguousarray(tr.arr[t0:t1]), np.ascontiguousarray(tr.now[t0:t1]), np.ascontiguousarray(tr.at[t0:t1]))
        tickets.append(g.run_host_async(*args, out, o, ttis_per_launch=7, traffic=traffic))
        keep.append((args, traffic, o))
        outs.append(out)
    for tk in tickets:
        g.wait(tk)
    got = {k: np.concatenate([x[k] for x in outs]) for k in outs[0]}
    check(c, (got, [g.get_state()], [g.get_buffers()]), want, tag="async")
    g.close()


@gpu
def test_profiles_with_different_arrivals():
    """P = 3 slice profiles, each with its own arrival spec (rs_synth_arrivals reads each cell's row)."""
    c = Case(9, CELLS["narrow"], B=6, T=60, seed=7900, nb=1)
    rng = np.random.default_rng(5)
    profs = [(c.w, c.p, c.u2s), (rng.dirichlet(np.ones(c.S)), c.p[::-1].copy(), c.u2s),
             (c.w[::-1].copy(), c.p, c.u2s)]
    cp = np.array([0, 1, 2, 2, 1, 0], dtype=np.int32)
    tr = Traffic(c, seed=9, n_profiles=3, cell_profile=cp)
    assert not np.array_equal(tr.pkt[0], tr.pkt[1]) or not np.array_equal(tr.q16[0], tr.q16[1])
    g = sched.Scheduler.from_profiles(9, profs, cp)
    g.enable_buffers(K, tr.backlogged)
    bounds = [25, 60]
    got = device_run(c, g, tr, bounds, 16)
    # one oracle per profile over its own cells
    for p in range(3):
        cells = np.flatnonzero(cp == p)
        o = OracleScheduler(9, profs[p][0], profs[p][1], c.u2s, len(cells))
        m = BufferModel(tr.backlogged[cells].shape, K, tr.backlogged[cells])
        act = c.active[:, cells]
        w_outs, w_states, w_bufs = closed_loop(o, m, c.ocqi[:, cells], c.draws[:, cells], c.dts, tr.arr[:, cells],
                                               tr.now, tr.at, active=act, bounds=bounds)
        for k, v in got[0].items():
            assert np.array_equal(v[:, cells], w_outs[k]), (p, k)
        for i in range(2):
            for k in ("avg_rate", "cum_bytes", "slice_offset"):
                assert np.array_equal(got[1][i][k][cells], w_states[i][k]), (p, i, k)
            for k in w_bufs[i]:
                assert np.array_equal(got[2][i][k][cells], w_bufs[i][k]), (p, i, k)
    g.close()


# ---- 3. two public paths agree --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("algo,nb", [(9, 1), (8, 2), (1, 1)])
def test_device_loop_equals_host_driven_loop(algo, nb):
    """The device closed loop == the same loop driven from the host through rs_set_queues, one TTI per call; 130 TTIs
    in one call == 10 calls of 13."""
    c = Case(algo, CELLS["narrow"], B=4, T=130, seed=8000 + algo + nb, nb=nb)
    tr = Traffic(c, seed=algo * 3 + nb)
    h = c.scheduler()
    want = closed_loop(h, tr.model(c), c.ocqi, c.draws, c.dts, tr.arr, tr.now, tr.at, active=c.active, bounds=[130])
    h.close()
    assert_drains_and_builds(want[0], tr)
    for bounds in ([130], list(range(13, 131, 13))):
        g = buffered(c, tr)
        got = host_run(c, g, tr, bounds, 16)
        check(c, (got[0], got[1][-1:], got[2][-1:]), want, tag=f"{len(bounds)} calls")
        g.close()


# ---- 4. hand-computed cases -----------------------------------------------------------------------------------------
def _one_cell(algo=9, nb=1, ups=(2, 2)):
    S = len(ups)
    u2s = np.repeat(np.arange(S), ups).astype(np.int32)
    p = np.zeros((S, 4), np.int32)
    p[:, 2] = 1
    g = sched.Scheduler(algo, np.full(S, 1.0 / S), p, u2s, 1, n_bearers=nb)
    return g, len(u2s)


def _cqi(U, v=10):
    return np.full((1, U, 64), v, np.uint8)


@gpu
def test_partial_head_keeps_its_timestamp_and_overflow_drops_whole_arrivals():
    g, U = _one_cell()
    g.enable_buffers(2)
    arr = np.zeros((1, U), np.int32)
    arr[0, 0] = 100000                       # far more than a TTI sends

    def sent():
        return int(g.get_state()["cum_bytes"][0, 0])

    o = g.step(_cqi(U), dt=0.001, arrivals=arr, now=1.0, arrival_time=0.9995)
    assert o["queue_out"][0, 0] == 100000 and o["hol_out"][0, 0] == 1.0 - 0.9995
    s1 = sent()
    assert 0 < s1 < 100000
    st = g.get_buffers()
    assert st["queued"][0, 0] == 100000 - s1 and st["n_records"][0, 0] == 1 and st["head_time"][0, 0] == 0.9995
    o = g.step(_cqi(U), dt=0.001, arrivals=arr, now=1.001, arrival_time=1.0005)   # a second record
    assert o["queue_out"][0, 0] == 200000 - s1
    assert o["hol_out"][0, 0] == 1.001 - 0.9995                                   # the partly sent head keeps its time
    s2 = sent()
    o = g.step(_cqi(U), dt=0.001, arrivals=arr, now=1.002, arrival_time=1.0015)   # K = 2 records held: dropped whole
    assert o["queue_out"][0, 0] == 200000 - s2
    st = g.get_buffers()
    assert st["dropped"][0, 0] == 100000 and st["queued"][0, 0] == 200000 - sent()
    assert st["n_records"][0, 0] == 2 and st["head_time"][0, 0] == 0.9995
    g.close()


@gpu
def test_backlogged_flags_and_id1_clamp():
    g, U = _one_cell(algo=1, ups=(4,))
    bl = np.zeros((1, U), bool)
    bl[0, 1] = True
    g.enable_buffers(4, bl)
    arr = np.zeros((1, U), np.int32)
    arr[0, 0] = 10                           # id 1 books its whole TBS to a flow, far above 10 bytes
    arr[0, 1] = 500                          # ignored: backlogged
    o = g.step(_cqi(U), dt=0.001, arrivals=arr, now=0.1, arrival_time=0.1)
    assert o["queue_out"][0, 1] == 100000000 and o["hol_out"][0, 1] == 0.0
    assert o["queue_out"][0, 0] == 10 and o["queue_out"][0, 2] == 0
    assert int(g.get_state()["cum_bytes"][0, 0]) > 10
    st = g.get_buffers()
    assert st["queued"][0, 0] == 0 and st["n_records"][0, 0] == 0 and st["queued"][0, 1] == 0
    g.close()


@gpu
def test_hol_never_negative_on_alpha_without_beta_slices():
    c = Case(9, CELLS["narrow"], B=3, T=60, seed=8100)
    c.p[:, 0], c.p[:, 1] = 1, 0             # alpha without beta everywhere: a negative delay would zero the metric
    tr = Traffic(c, seed=4)
    want = oracle_loop(c, tr, [60])
    g = buffered(c, tr)
    got = host_run(c, g, tr, [60], 16)
    assert (got[0]["hol_out"] >= 0).all()
    check(c, got, want)
    g.close()


# ---- 5. generator and log writer -----------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("nb", [1, 2])
def test_synth_arrivals_matches_workload(nb):
    import torch
    c = Case(9, CELLS["wide"], B=3, T=9, seed=1, nb=nb)
    cp = np.array([1, 0, 1], np.int32)
    profs = [(c.w, c.p, c.u2s), (c.w, c.p, np.roll(c.u2s, 7))]
    g = sched.Scheduler.from_profiles(9, profs, cp, n_bearers=nb)
    pkt = np.array([[0, 1500] * (c.S // 2) + [300] * (c.S % 2), [40] * c.S], np.int32)
    q16 = np.array([np.arange(c.S) * 40000, [65536 * 3 + 1] * c.S], np.int32)
    want = workload.synth_arrivals(99, 5, 3, 17, 9, np.stack([p[2] for p in profs]), pkt, q16, n_bearers=nb, cell_profile=cp)
    d = torch.empty(want.shape, dtype=torch.int32).cuda()
    g.synth_arrivals(99, 5, 17, 9, pkt, q16, d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy(), want)
    assert (want > 0).any() and (want == 0).any()
    g.close()


@gpu
def test_log_writer_from_queue_out():
    """queue_out / hol_out fed to rs_log_set_queues give the text of the oracle-driven loop."""
    c = Case(9, CELLS["narrow"], B=2, T=40, seed=8200, nb=2)
    tr = Traffic(c, seed=8)
    want = oracle_loop(c, tr, [40])
    g = buffered(c, tr)
    got = host_run(c, g, tr, [40], 7)

    def log(outs):
        lg = sched.LogWriter(9, c.u2s, c.S, n_bearers=2)
        for t in range(c.T):
            lg.tti(100 + t, c.ocqi[t, 1], outs["rbg_to_ue"][t, 1], outs["tbs_bits"][t, 1], outs["final_cqi"][t, 1],
                   outs["slice_target"][t, 1], outs["slice_quota"][t, 1], queue=outs["queue_out"][t, 1],
                   hol=outs["hol_out"][t, 1])
        return lg.stdout, lg.stderr

    a, b = log(got[0]), log(want[0])
    assert a == b and re.search(r"hol_delay: 0\.0\d", a[1])
    g.close()


# ---- 6. argument checks ---------------------------------------------------------------------------------------------
@gpu
def test_argument_checks():
    g, U = _one_cell(nb=2)
    cqi, arr = _cqi(U), np.zeros((1, U, 2), np.int32)
    for k in (-1, 65537):
        with pytest.raises(sched.RsError, match="max_records"):
            g.enable_buffers(k)
    g.enable_buffers(4)
    with pytest.raises(sched.RsError, match="rs_set_queues"):
        g.step(cqi, queue=np.ones((1, U, 2), np.int32))
    with pytest.raises(sched.RsError, match="rs_set_traffic"):
        g.step(cqi)
    with pytest.raises(sched.RsError, match="arrival_time"):
        g.step(cqi, arrivals=arr, now=1.0, arrival_time=1.5)
    g.step(cqi, arrivals=arr, now=1.0)
    with pytest.raises(sched.RsError, match="before the previous"):
        g.step(cqi, arrivals=arr, now=0.999)
    g.step(cqi, arrivals=arr, now=1.0)          # the same time again is allowed
    with pytest.raises(sched.RsError, match="rs_step_cell"):
        g.step_cell(cqi)
    g.reset_state()                              # forgets the last now
    g.step(cqi, arrivals=arr, now=0.5)
    g.enable_buffers(0)                          # off: rs_set_queues works again
    with pytest.raises(sched.RsError, match="no buffers"):
        g.get_buffers()
    g.step(cqi, queue=np.ones((1, U, 2), np.int32))
    g.close()

"""Slice profiles (rs_create_profiles): cells with different slice configurations in one batch, against the CPU oracle.

Contract: cell b is scheduled bit for bit as a one-profile handle built from profile cell_profile[b] schedules it.  The
oracle side therefore runs one OracleScheduler per profile over the cells of that profile (id 11: each cell's rand()
row cut to that profile's own stride, 300 x its largest slice) and hands every cell's state on at each call boundary,
which is also how a cell changes profile (rs_set_cell_profiles).  Every output of every TTI and the whole state at
every call boundary are compared bit for bit."""
import ctypes as C

import numpy as np
import pytest

from oracle.pyoracle import OracleScheduler
from radiosaber_b200 import sched, workload
from tests.test_kernel_paths_gpu import CELLS, IDS, NVS, THREADS, TRANSPORT, Case, _env, _equal_runs

gpu = pytest.mark.gpu

# per width: profiles of the same S and U that differ in UEs per slice (and so in the largest slice: the metric-table
# chunks, m_cap, id 7's / 11's per-user scratch and id 11's rand() stride); the last one is assigned to no cell
UPS = {"narrow": [CELLS["narrow"], [8, 4, 5, 2, 7, 1, 3], [1, 1, 1, 1, 1, 1, 24], [4, 4, 4, 4, 4, 5, 5]],
       "wide": [CELLS["wide"], [70, 30, 45, 40, 38, 50, 42, 35, 48, 44, 39, 2], CELLS["wide"][::-1],
                [43] + [40] * 11]}
# irregular: neither blocks nor round-robin; profile 3 unused
CP = [2, 0, 0, 1, 2, 2, 0, 1, 2]
# narrow cells of 49 UEs: no profile gets direct metrics unless asked to (slices of < 8 UEs in profile 0)
FORCE_DIRECT_UPS = [[7] * 7, [5, 7, 7, 7, 7, 7, 9], [1, 1, 7, 7, 7, 7, 19], [9, 8, 8, 8, 8, 4, 4]]
STATE_KEYS = ("avg_rate", "tx_bytes", "cum_bytes", "cum_rbs", "slice_offset", "nvs_ewma")


def _params(rng, S):
    p = np.zeros((S, 4), dtype=np.int32)
    p[:, 0] = rng.integers(0, 2, S)
    p[:, 1] = rng.integers(0, 2, S)
    p[:, 2] = rng.choice([0, 1, 1, 2], S)
    p[:, 3] = rng.integers(0, 2, S)
    return p


class ProfCase(Case):
    """Case's seeded inputs (built on the profile with the largest slice, so that its rand() stride is the handle's)
    with P profiles: their own weights, alpha / beta / epsilon / psi and UEs per slice."""

    def __init__(self, algo, ups_list, cp, T, seed, same=False, neg_hol=True, **kw):
        big = max(range(len(ups_list)), key=lambda k: max(ups_list[k]))
        super().__init__(algo, ups_list[big], len(cp), T, seed, **kw)
        rng = np.random.default_rng(seed + 17)
        self.profiles = []
        for k, ups in enumerate(ups_list):
            assert len(ups) == self.S and sum(ups) == self.U
            w, p = (self.w, self.p) if (k == big or same) else (rng.dirichlet(np.ones(self.S)), _params(rng, self.S))
            self.profiles.append((w, p, np.repeat(np.arange(self.S), ups).astype(np.int32)))
        self.cp = np.asarray(cp, dtype=np.int32)
        if self.hol is not None:
            # negative delays are defined for alpha-without-beta slices only (an empty prioritised bearer, rs_set_queues):
            # re-drawn per cell on the alpha-only slices of the cell's own profile
            self.hol = np.abs(self.hol)
            if neg_hol and self.nb == 1 and algo in TRANSPORT:
                draw = np.random.default_rng(seed + 29).random(self.hol.shape) < 0.15
                for b in range(self.B):
                    _, p, u2s = self.profiles[self.cp[b]]
                    gate_only = ((p[:, 0] != 0) & (p[:, 1] == 0))[u2s]
                    self.hol[:, b] = np.where(draw[:, b] & gate_only, -1.0, self.hol[:, b])

    def scheduler(self, cp=None, **env):
        with _env(**env):
            g = sched.Scheduler.from_profiles(self.algo, self.profiles, self.cp if cp is None else cp,
                                              cqi_per_rb=self.layout, **self.cfg())
        assert g.n_profiles == len(self.profiles)
        assert g.rand_stride == (self.stride if self.algo in TRANSPORT + (11,) else 0)
        if self.trace:
            g.set_traces(self.traces, self.ue_trace)
        return g

    def stride_of(self, k):
        return 300 * int(np.bincount(self.profiles[k][2]).max()) if self.algo == 11 else self.stride

    def oracle(self, bounds, cps=None):
        """Outputs [T][B][...] and the state after every call; cps[i] = the assignment in force during call i."""
        T, B = self.T, self.B
        cps = [self.cp] * len(bounds) if cps is None else cps
        o0 = OracleScheduler(self.algo, *self.profiles[0], B, cqi_per_rb=1 if self.layout == 1 else 0, **self.cfg())
        state = o0.get_state()   # every cell's state, handed from call to call and from profile to profile
        outs, states, t0 = {}, [], 0
        for t1, cp in zip(bounds, cps):
            for k in range(len(self.profiles)):
                idx = np.flatnonzero(np.asarray(cp) == k)
                if idx.size == 0:
                    continue
                o = OracleScheduler(self.algo, *self.profiles[k], idx.size, cqi_per_rb=1 if self.layout == 1 else 0,
                                    n_threads=8, **self.cfg())
                o.set_state(**{n: state[n][idx] for n in STATE_KEYS})
                n = self.stride_of(k)
                for t in range(t0, t1):
                    kw = {} if self.queue is None else {"queue": self.queue[t][idx], "hol": self.hol[t][idx]}
                    r = o.step(self.ocqi[t][idx], self.draws[t][idx][:, :n], dt=float(self.dts[t]),
                               active=None if self.active is None else self.active[t][idx], want_aux=True, **kw)
                    for name, v in r.items():
                        if name not in outs:
                            outs[name] = np.zeros((T, B) + v.shape[1:], v.dtype)
                        outs[name][t, idx] = v
                st = o.get_state()
                for name in STATE_KEYS:
                    state[name][idx] = st[name]
            states.append({n: v.copy() for n, v in state.items()})
            t0 = t1
        return outs, states

    def run_host(self, g, bounds, tpl, cps=None):
        """As Case.run_host; cps[i] (i > 0) is set with rs_set_cell_profiles before call i."""
        outs, states, t0 = [], [], 0
        for i, t1 in enumerate(bounds):
            if cps is not None and i > 0:
                g.set_cell_profiles(cps[i])
            kw = dict(active=self._sl(self.active, t0, t1), want_aux=True, ttis_per_launch=tpl,
                      queue=self._sl(self.queue, t0, t1), hol=self._sl(self.hol, t0, t1))
            draws, dts = self.draws[t0:t1], self.dts[t0:t1]
            if self.trace:
                outs.append(g.run_traces_host(self.rows[t0:t1], draws, dts, **kw))
            else:
                outs.append(g.run_host(self.slabs[t0:t1], draws, dts, **kw))
            states.append(g.get_state())
            t0 = t1
        return {k: np.concatenate([x[k] for x in outs]) for k in outs[0]}, states


def _stats_statement(c, st, cp):
    """uint64 [P][4][S] computed on the host from get_state(): per profile, its cells, its ue_to_slice."""
    P, S = len(c.profiles), c.S
    want = np.zeros((P, 4, S), dtype=np.uint64)
    cb = st["cum_bytes"].reshape(c.B, c.U, -1)
    cr = st["cum_rbs"].reshape(c.B, c.U, -1)
    for b in range(c.B):
        u2s = c.profiles[cp[b]][2]
        for u in range(c.U):
            for k in range(cb.shape[2]):
                q = cb[b, u, k] >> np.uint64(10)
                want[cp[b], :, u2s[u]] += np.array([cb[b, u, k], cr[b, u, k], q, q * q], dtype=np.uint64)
    return want


# ---- 1. the matrix: every id x both CTA widths x streamed / trace CQI x backlogged / queue-aware --------------------
@gpu
@pytest.mark.parametrize("queue", [False, True])
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("algo", IDS)
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_profile_matrix(width, algo, trace, queue):
    c = ProfCase(algo, UPS[width], CP, T=20, seed=500 * IDS.index(algo) + 50 * (width == "wide") + 2 * trace + queue,
                 trace=trace, queue=queue, layout=2 if (trace and not queue) else 0)
    g = c.scheduler()
    assert sched.lib().rs_threads_per_cta(g._h) == THREADS[width]
    assert sched.lib().rs_n_profiles(g._h) == 4
    bounds = [9, 20]
    c.check(c.run_host(g, bounds, 5), c.oracle(bounds))
    g.close()


@gpu
@pytest.mark.parametrize("algo", [7, 8, 9, 10, 11, 101, 103])
def test_profile_matrix_two_bearers(algo):
    c = ProfCase(algo, UPS["narrow"], CP, T=16, seed=900 + algo, nb=2)
    g = c.scheduler()
    bounds = [7, 16]
    c.check(c.run_host(g, bounds, 4), c.oracle(bounds))
    g.close()


# ---- 2. the headline cell keeps its compile-time-shape kernel under a weight / scheduler sweep --------------------
@gpu
@pytest.mark.parametrize("layout", [0, 2])
@pytest.mark.parametrize("algo", [7, 8, 9, 10, 11, 101, 103])
def test_fixed_shape_with_twenty_profiles(algo, layout):
    rng = np.random.default_rng(40 + algo + layout)
    ups = [[5] * 20] * 20
    cp = rng.integers(0, 20, 53)
    cp[:20] = rng.permutation(20)
    c = ProfCase(algo, ups, cp, T=12, seed=3000 + algo * 3 + layout, layout=layout)
    g = c.scheduler()
    assert sched.lib().rs_fixed_shape(g._h) >= 0
    bounds = [5, 12]
    want = c.oracle(bounds)
    c.check(c.run_host(g, bounds, 4), want)
    g.close()
    # one profile's UEs remapped: the general kernel, same results
    c.profiles[7] = (c.profiles[7][0], c.profiles[7][1], np.roll(c.profiles[7][2], 1))
    g = c.scheduler()
    assert sched.lib().rs_fixed_shape(g._h) == -1
    c.check(c.run_host(g, bounds, 4), c.oracle(bounds), tag="remapped")
    g.close()


# ---- 3. identical profiles are one profile ------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("algo", IDS)
def test_identical_profiles_equal_one_profile(algo):
    for width in ("narrow", "wide"):
        c = ProfCase(algo, [CELLS[width]] * 3, CP[:7], T=12, seed=60 + algo, same=True, queue=True)
        one = sched.Scheduler(algo, c.w, c.p, c.u2s, c.B, **c.cfg())
        many = c.scheduler()
        for f in ("rs_smem_bytes", "rs_fixed_shape", "rs_direct_metric", "rs_threads_per_cta", "rs_rand_draws_per_cell_tti"):
            assert getattr(sched.lib(), f)(one._h) == getattr(sched.lib(), f)(many._h), (width, f)
        bounds = [5, 12]
        a, b = c.run_host(one, bounds, 3), c.run_host(many, bounds, 3)
        _equal_runs(a, b, width)
        st = many.get_stats()
        assert st.shape == (3, 4, c.S)
        assert np.array_equal(st.sum(axis=0), one.get_stats())
        assert np.array_equal(st, _stats_statement(c, many.get_state(), c.cp))
        one.close()
        many.close()


# ---- 4. the launch paths --------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("algo", [8, 9, 10, 101, 103])
def test_direct_metric_with_profiles(algo):
    """Big slices: the direct per-slice argmax stages the cell's own Epow rows.  The wide cells pick it on their own; 49
    UEs in slices of at most 7 to 19 (two or more metric-table chunks) take it with RS_FORCE_DIRECT."""
    for ups, env in ((UPS["wide"], {}), (FORCE_DIRECT_UPS, {"RS_FORCE_DIRECT": 1})):
        c = ProfCase(algo, ups, CP, T=10, seed=70 + algo, queue=True, active=False)
        g = c.scheduler(**env)
        assert sched.lib().rs_direct_metric(g._h) == 1, env
        bounds = [4, 10]
        c.check(c.run_host(g, bounds, 3), c.oracle(bounds), tag=str(env))
        g.close()


@gpu
@pytest.mark.parametrize("algo", IDS)
def test_paths_no_stage_parts_device(algo):
    c = ProfCase(algo, UPS["narrow"], CP, T=14, seed=80 + algo, queue=True)
    bounds = [6, 14]
    want = c.oracle(bounds)
    for env in ({"RS_NO_STAGE": 1}, {"RS_PARTS": 3}):
        g = c.scheduler(**env)
        c.check(c.run_host(g, bounds, 4), want, tag=str(env))
        if "RS_PARTS" in env:
            g.reset_state()
            c.check(c.run_device(g, bounds, 4), want, tag="device")
        g.close()


@gpu
@pytest.mark.parametrize("algo", [1, 9, 11, 103])
def test_multi_tti_launches_with_queues(algo):
    c = ProfCase(algo, UPS["narrow"], CP, T=70, seed=90 + algo, queue=True)
    bounds = [33, 70]
    want = c.oracle(bounds)
    for tpl in (1, 64):
        g = c.scheduler()
        c.check(c.run_host(g, bounds, tpl), want, tag=tpl)
        g.close()


@gpu
@pytest.mark.parametrize("algo", [7, 9, 10, 11])
def test_step_cell_with_profiles(algo):
    """rs_step_cell: the caller's rates and slice state travel with the inputs."""
    c = ProfCase(algo, UPS["narrow"], CP, T=6, seed=110 + algo, queue=True)
    g = c.scheduler()
    want = c.oracle(list(range(1, c.T + 1)))
    avg = np.full((c.B, c.U), 100000.0)
    ss = np.zeros((c.B, c.S))
    for t in range(c.T):
        got = g.step_cell(c.ocqi[t], c.draws[t], dt=float(c.dts[t]), active=c.active[t], queue=c.queue[t], hol=c.hol[t],
                          avg_rate=avg, slice_state=ss)
        for k, v in got.items():
            if k in ("alloc_ue", "alloc_rbg"):
                continue
            assert np.array_equal(v, want[0][k][t]), (t, k)
        assert np.array_equal(avg, want[1][t]["avg_rate"]), t
        assert np.array_equal(ss, want[1][t]["nvs_ewma" if algo in NVS else "slice_offset"]), t
    g.close()


@gpu
def test_two_async_calls_in_flight():
    c = ProfCase(9, UPS["narrow"], CP, T=16, seed=120, active=False)
    g = c.scheduler()
    want = c.oracle([8, 16])
    tickets, res = [], []
    for t0, t1 in ((0, 8), (8, 16)):
        out, o = g._host_outputs(t1 - t0, True)
        args = (np.ascontiguousarray(c.slabs[t0:t1]), g._draws(c.draws[t0:t1], (t1 - t0, c.B)),
                np.ascontiguousarray(c.dts[t0:t1]))
        tickets.append(g.run_host_async(*args, out, o, 4))
        res.append((out, o, args))
    for tk in tickets:
        g.wait(tk)
    for k in res[0][0]:
        got = np.concatenate([res[0][0][k], res[1][0][k]])
        assert np.array_equal(got, want[0][k]), k
    assert np.array_equal(g.get_state()["avg_rate"], want[1][-1]["avg_rate"])
    g.close()


# ---- 5. a new assignment between calls ---------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("algo", IDS)
def test_set_cell_profiles_between_calls(algo):
    c = ProfCase(algo, UPS["narrow"], CP, T=18, seed=130 + algo, queue=True, neg_hol=False)
    cps = [c.cp, np.array([3, 1, 0, 0, 3, 2, 1, 1, 0], dtype=np.int32), np.array([1, 3, 2, 1, 1, 0, 2, 3, 3], dtype=np.int32)]
    bounds = [6, 12, 18]
    g = c.scheduler()
    c.check(c.run_host(g, bounds, 4, cps=cps), c.oracle(bounds, cps=cps))
    assert np.array_equal(g.get_stats(), _stats_statement(c, g.get_state(), cps[-1]))
    g.close()


@gpu
def test_set_cell_profiles_right_after_an_async_call():
    """The new assignment waits for the call in flight: its TTIs still run under the old one."""
    c = ProfCase(9, UPS["narrow"], CP, T=16, seed=140, active=False)
    cps = [c.cp, np.array([1, 2, 1, 0, 3, 3, 2, 0, 1], dtype=np.int32)]
    want = c.oracle([8, 16], cps=cps)
    g = c.scheduler()
    out, o = g._host_outputs(8, True)
    args = (np.ascontiguousarray(c.slabs[:8]), g._draws(c.draws[:8], (8, c.B)), np.ascontiguousarray(c.dts[:8]))
    ticket = g.run_host_async(*args, out, o, 2)
    g.set_cell_profiles(cps[1])
    g.wait(ticket)
    second = g.run_host(c.slabs[8:], c.draws[8:], c.dts[8:], want_aux=True, ttis_per_launch=4)
    for k in out:
        assert np.array_equal(np.concatenate([out[k], second[k]]), want[0][k]), k
    st = g.get_state()
    for k in ("avg_rate", "tx_bytes", "cum_bytes", "cum_rbs", "slice_offset"):
        assert np.array_equal(st[k], want[1][-1][k]), k
    g.close()


# ---- 6. statistics ------------------------------------------------------------------------------------------------
@gpu
def test_stats_per_profile_and_single_rank_reduce():
    import os
    import torch  # noqa: F401  -- before librs_nccl.so (see tests/test_host_api_gpu.py::_nccl)
    from tests.helpers import ROOT
    c = ProfCase(9, UPS["narrow"], CP, T=30, seed=150, queue=True)
    g = c.scheduler()
    c.run_host(g, [30], 8)
    st = g.get_stats()
    want = _stats_statement(c, g.get_state(), c.cp)
    assert st.shape == (4, 4, c.S) and np.array_equal(st, want) and st[3].sum() == 0 and st[0, 0].sum() > 0
    L = C.CDLL(os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so"))
    L.rs_nccl_last_error.restype = C.c_char_p
    L.rs_reduce_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    L.rs_comm_destroy.argtypes = [C.c_void_p]
    uid = (C.c_uint8 * 128)()
    assert L.rs_comm_unique_id(uid) == 0, L.rs_nccl_last_error()
    comm = C.c_void_p()
    assert L.rs_comm_init_rank(1, 0, uid, 0, C.byref(comm)) == 0, L.rs_nccl_last_error()
    red = np.zeros_like(st)
    assert L.rs_reduce_stats(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, L.rs_nccl_last_error()
    L.rs_comm_destroy(comm)
    assert np.array_equal(red, st)
    g.close()

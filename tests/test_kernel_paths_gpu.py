"""Every path of the TTI kernel the C ABI can launch, against the CPU oracle.

The other parity tests sit on a few rails (64 RBGs, one TTI per launch whenever queues are finite, streamed CQI with
queues or two bearers).  Here the same seeded inputs go through the oracle TTI by TTI and through one device entry
point: both CTA widths x all eight ids x streamed / trace-replayed CQI x backlogged / queue-aware x the three CQI
layouts, two bearers, multi-TTI launches with queues, device-resident queues, CQI staging on and off, part-batches
and the RBG counts of the LTE-Sim bands.  Every output of every TTI and the whole state at every call boundary are
compared bit for bit.

The matrix table below names every (width, id, CQI source, queue-aware) instantiation of rs_tti_kernel; a CPU test
reads rs_kernels.cu and fails when an instantiation is missing from it."""
import contextlib
import os
import re

import numpy as np
import pytest

from oracle import trace_ingest as ti
from oracle.pyoracle import OracleScheduler
from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

gpu = pytest.mark.gpu

IDS = (1, 7, 8, 9, 10, 11, 101, 103)
TRANSPORT = (8, 9, 10, 101, 103)
NVS = (7, 11)
# ~30 UEs in uneven slices (128 threads); >= 480 UEs with a 1-UE and a 60-UE slice (512 threads)
CELLS = {"narrow": [3, 1, 7, 2, 5, 4, 8], "wide": [1, 60, 45, 40, 38, 50, 42, 35, 48, 44, 39, 41]}
THREADS = {"narrow": 128, "wide": 512}
# (width, id, trace replay, queue-aware): one entry per general instantiation of rs_tti_kernel (rs_kernels.cu)
MATRIX = [(w, a, tr, q) for w in ("narrow", "wide") for a in IDS for tr in (False, True) for q in (False, True)]
# (n_rbs, rbg_size) of LTE-Sim's 6/15/25/50/75/100-RB bands trimmed to whole RBGs the way the plug-in does
# (host/rs_gpu_scheduler.h), with RBG sizes of 36.213 Table 7.1.6.1-1 (1 up to 10 RBs, 2 up to 26, 3 up to 63, 4 up
# to 110; assumed, the reference's get_rbg_size is documented for 111..512 RBs only), plus 256 / 504 RBs in RBGs of 8
# and 64 RBGs of one RB
BANDS = [(6, 1), (14, 2), (24, 2), (48, 3), (72, 4), (100, 4), (256, 8), (504, 8), (64, 1)]


@contextlib.contextmanager
def _env(**kv):
    """Environment switches rs_create reads (set for the handle's creation only)."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


class Case:
    """Seeded inputs of one run: slices with random alpha / beta / epsilon / psi, T TTIs of CQI (streamed slabs or
    trace replay with rows -1 before the first report and some UEs on trace -1), rand() draws, an active mask with an
    all-idle cell 0 and a cell 1 where only slice 1 has data, and optionally finite queues with head-of-line delays."""

    def __init__(self, algo, ups, B, T, seed, n_rbs=512, rbg=8, layout=0, trace=False, queue=False, nb=1, refresh=1,
                 active=True):
        rng = np.random.default_rng(seed)
        self.algo, self.B, self.T, self.layout, self.trace, self.nb, self.refresh = algo, B, T, layout, trace, nb, refresh
        self.R, self.rbg, self.G = n_rbs, rbg, n_rbs // rbg
        S = self.S = len(ups)
        self.u2s = np.repeat(np.arange(S), ups).astype(np.int32)
        U = self.U = len(self.u2s)
        self.w = rng.dirichlet(np.ones(S))
        p = np.zeros((S, 4), dtype=np.int32)
        p[:, 0] = rng.integers(0, 2, S)
        p[:, 1] = rng.integers(0, 2, S)
        p[:, 2] = rng.choice([0, 1, 1, 2], S)
        p[:, 3] = rng.integers(0, 2, S)
        self.p = p
        G, R = self.G, n_rbs
        if trace:
            n_tr, n_rows = 5, 9
            if layout == 1:
                self.traces = rng.integers(1, 16, (n_tr, n_rows, R)).astype(np.uint8)
            else:
                self.traces = np.repeat(workload.histogram_cqi(rng, (n_tr, n_rows, G)), rbg, axis=2)
            self.ue_trace = rng.integers(-1, n_tr, (B, U)).astype(np.int32)
            self.rows = np.repeat(rng.integers(0, n_rows, T // 5 + 1), 5)[:T].astype(np.int32)
            self.rows[:3] = -1
            otab = self.traces if layout == 1 else self.traces[:, :, ::rbg]
            self.ocqi = np.stack([ti.cqi_at(otab, self.ue_trace, int(r)) for r in self.rows])
        else:
            slabs = workload.synth_cqi(seed, 0, B, 0, -(-T // refresh), U, G)   # "tti" e of the generator = epoch e
            if layout == 1:
                slabs = np.clip(np.repeat(slabs, rbg, axis=-1).astype(np.int64) + rng.integers(-1, 2, slabs.shape[:-1] + (R,)),
                                1, 15).astype(np.uint8)
            self.ocqi = slabs[np.arange(T) // refresh]
            self.slabs = sched.pack_cqi(slabs) if layout == 2 else slabs
        self.stride = 300 * max(ups) if algo == 11 else 2
        self.draws = workload.synth_rand_draws(seed, 0, B, 0, T, S, self.stride)
        self.now, self.dts = workload.tti_clock(T)
        self.active = None
        if active:
            self.active = (rng.random((T, B, U)) < 0.85).astype(np.uint8)
            self.active[:, 0] = 0
            if B > 1:
                self.active[:, 1, self.u2s != 1] = 0
        self.queue = self.hol = None
        if queue or nb == 2:
            per = (T, B, U) if nb == 1 else (T, B, U, 2)
            kind = rng.random(per)
            self.queue = np.where(kind < 0.15, 0, np.where(kind < 0.6, rng.integers(20, 20000, per), 100000000)).astype(np.int32)
            self.hol = np.where(rng.random(per) < 0.1, 0.0, rng.random(per) * 0.08)
            if nb == 1 and algo in TRANSPORT:
                # negative delays only where the ABI defines them: alpha-without-beta slices (rs_set_queues)
                gate_only = ((p[:, 0] != 0) & (p[:, 1] == 0))[self.u2s]
                self.hol = np.where((rng.random(per) < 0.1) & gate_only, -1.0, self.hol)

    def cfg(self):
        return dict(n_rbs=self.R, rbg_size=self.rbg, n_bearers=self.nb)

    def scheduler(self, **env):
        with _env(**env):
            g = sched.Scheduler(self.algo, self.w, self.p, self.u2s, self.B, cqi_per_rb=self.layout, **self.cfg())
        assert g.rand_stride == (self.stride if self.algo in TRANSPORT + (11,) else 0)
        if self.trace:
            g.set_traces(self.traces, self.ue_trace)
        return g

    def oracle(self, bounds):
        """Outputs of every TTI ([T][B][...]) and the state after the last TTI of every call."""
        o = OracleScheduler(self.algo, self.w, self.p, self.u2s, self.B, cqi_per_rb=1 if self.layout == 1 else 0,
                            n_threads=8, **self.cfg())
        outs, states = [], []
        for t in range(self.T):
            kw = {} if self.queue is None else {"queue": self.queue[t], "hol": self.hol[t]}
            outs.append(o.step(self.ocqi[t], self.draws[t], dt=float(self.dts[t]),
                               active=None if self.active is None else self.active[t], want_aux=True, **kw))
            if t + 1 in bounds:
                states.append(o.get_state())
        return {k: np.stack([x[k] for x in outs]) for k in outs[0]}, states

    def _sl(self, a, t0, t1):
        return None if a is None else a[t0:t1]

    def run_host(self, g, bounds, tpl):
        """rs_run_host / rs_run_traces_host, one call per [bounds[i-1], bounds[i])."""
        outs, states, t0 = [], [], 0
        for t1 in bounds:
            kw = dict(active=self._sl(self.active, t0, t1), want_aux=True, ttis_per_launch=tpl,
                      queue=self._sl(self.queue, t0, t1), hol=self._sl(self.hol, t0, t1))
            draws, dts = self.draws[t0:t1], self.dts[t0:t1]
            if self.trace:
                outs.append(g.run_traces_host(self.rows[t0:t1], draws, dts, **kw))
            else:
                assert t0 % self.refresh == 0
                slabs = self.slabs[t0 // self.refresh:-(-t1 // self.refresh)]
                outs.append(g.run_host(slabs, draws, dts, cqi_refresh=self.refresh, **kw))
            states.append(g.get_state())
            t0 = t1
        return {k: np.concatenate([x[k] for x in outs]) for k in outs[0]}, states

    def run_device(self, g, bounds, tpl):
        """rs_run_device / rs_run_traces_device with every input, queues and delays included, in torch tensors."""
        import torch

        def dev(a):
            return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()

        T, B, U, S, G = self.T, self.B, self.U, self.S, self.G
        out = {"rbg_to_ue": torch.empty((T, B, G), dtype=torch.int16), "tbs_bits": torch.empty((T, B, U), dtype=torch.int32),
               "mcs": torch.empty((T, B, U), dtype=torch.uint8), "final_cqi": torch.empty((T, B, U), dtype=torch.uint8)}
        if self.algo in TRANSPORT:
            out["slice_target"] = torch.empty((T, B, S), dtype=torch.int32)
            out["slice_quota"] = torch.empty((T, B, S), dtype=torch.int32)
        if self.algo in NVS:
            out["nvs_slice"] = torch.empty((T, B), dtype=torch.int32)
        if self.algo == 10:
            out["alloc_n"] = torch.empty((T, B), dtype=torch.int32)
            out["alloc_ue"] = torch.empty((T, B, 2 * G), dtype=torch.int16)
            out["alloc_rbg"] = torch.empty((T, B, 2 * G), dtype=torch.int16)
        out = {k: v.cuda() for k, v in out.items()}
        d_draws, d_act, d_q, d_h = dev(self.draws), dev(self.active), dev(self.queue), dev(self.hol)
        d_slabs = None if self.trace else dev(self.slabs)

        def ptr(a, t):
            return 0 if a is None else a[t].data_ptr()

        states, t0 = [], 0
        for t1 in bounds:
            n = t1 - t0
            kw = dict(d_out={k: v[t0].data_ptr() for k, v in out.items()}, d_active=ptr(d_act, t0),
                      active_tti_stride=B * U, ttis_per_launch=tpl, d_queue=ptr(d_q, t0), d_hol=ptr(d_h, t0))
            r2 = ptr(d_draws, t0) if g.rand_stride else 0
            if self.trace:
                g.run_traces_device(n, self.rows[t0:t1], r2, self.dts[t0:t1], **kw)
            else:
                assert t0 % self.refresh == 0
                g.run_device(n, ptr(d_slabs, t0 // self.refresh), d_slabs[0].numel(), r2, self.dts[t0:t1],
                             cqi_refresh=self.refresh, **kw)
            g.sync()
            states.append(g.get_state())
            t0 = t1
        return {k: v.cpu().numpy() for k, v in out.items()}, states

    def check(self, got, want, tag=""):
        outs, states = got
        w_outs, w_states = want
        for k, v in outs.items():
            if k in ("alloc_ue", "alloc_rbg"):   # the grant list: alloc_n entries per cell-TTI
                for t, b in np.ndindex(self.T, self.B):
                    n = int(w_outs["alloc_n"][t, b])
                    assert np.array_equal(v[t, b, :n], w_outs[k][t, b, :n]), (tag, k, t, b)
                continue
            bad = np.argwhere(v != w_outs[k])
            assert bad.size == 0, (tag, k, bad[:5].tolist())
        keys = ["avg_rate", "tx_bytes", "cum_bytes", "cum_rbs"]
        keys += ["slice_offset"] if self.algo in TRANSPORT else (["nvs_ewma"] if self.algo in NVS else [])
        assert len(states) == len(w_states)
        for i, (sa, sb) in enumerate(zip(states, w_states)):
            for k in keys:
                assert np.array_equal(sa[k], sb[k]), (tag, "state", i, k)


def _equal_runs(a, b, tag):
    for k in a[0]:
        assert np.array_equal(a[0][k], b[0][k]), (tag, k)
    for sa, sb in zip(a[1], b[1]):
        for k in sa:
            assert np.array_equal(sa[k], sb[k]), (tag, "state", k)


# ---- 1. the instantiation matrix ---------------------------------------------------------------------------------
def _kernel_picks():
    """{(width, id, trace, queue)} of the general rs_tti_kernel instantiations rs_kernels.cu holds: per translation unit
    the ids of its `case N` labels and of its `default`, each under the four (trace, queue) picks of RS_TTI_PICK."""
    src = open(os.path.join(ROOT, "radiosaber_b200", "csrc", "rs_kernels.cu")).read()
    pick = re.search(r"#define RS_TTI_PICK\(A\)(.*?)\n\n", src, re.S).group(1)
    combos = {(m.group(1) == "true", m.group(2) == "true")
              for m in re.finditer(r"rs_tti_kernel<A, (true|false), (true|false)>", pick)}
    assert combos == {(tr, q) for tr in (False, True) for q in (False, True)}, pick
    wide_tus = {int(x) for x in re.findall(r"RS_TU == (\d)", re.search(r"#if (RS_TU == \d[^\n]*)\n#define RS_NS rsw", src).group(1))}
    assert wide_tus == {3, 4}
    found = set()
    blocks = re.findall(r"#(?:el)?if ((?:RS_TU == \d(?: \|\| )?)+)\s*\nconst void\* RS_CAT\(rs_kernel_tu, RS_TU\)\(int algo, bool trace, "
                        r"bool queue\) \{(.*?)\n\}", src, re.S)
    assert len(blocks) == 2, blocks
    for cond, body in blocks:
        ids = [int(x) for x in re.findall(r"case (\d+): return RS_TTI_PICK\(\1\);", body)]
        ids += [int(x) for x in re.findall(r"default: return RS_TTI_PICK\((\d+)\);", body)]
        assert len(ids) == len(re.findall(r"RS_TTI_PICK", body)), body
        for tu in (int(x) for x in re.findall(r"RS_TU == (\d)", cond)):
            for a in ids:
                for tr, q in combos:
                    found.add(("wide" if tu in wide_tus else "narrow", a, tr, q))
    return found


def test_matrix_names_every_kernel_instantiation():
    """CPU: a new instantiation in rs_kernels.cu cannot land without an entry in MATRIX (and so a case below)."""
    picks = _kernel_picks()
    assert len(picks) == 64
    assert picks == set(MATRIX), (sorted(picks - set(MATRIX)), sorted(set(MATRIX) - picks))


def _check_width(g, width):
    assert sched.lib().rs_threads_per_cta(g._h) == THREADS[width]
    assert sched.lib().rs_fixed_shape(g._h) == -1


@gpu
@pytest.mark.parametrize("layout", [0, 1, 2])
@pytest.mark.parametrize("width,algo,trace,queue", MATRIX)
def test_instantiation_matrix(width, algo, trace, queue, layout):
    """30 TTIs in launches of 7, two calls (state compared at both boundaries)."""
    c = Case(algo, CELLS[width], B=4, T=30, seed=1000 * IDS.index(algo) + 100 * (width == "wide") + 10 * layout + 2 * trace + queue, layout=layout,
             trace=trace, queue=queue)
    g = c.scheduler()
    _check_width(g, width)
    bounds = [16, 30]
    c.check(c.run_host(g, bounds, 7), c.oracle(bounds))
    g.close()


@gpu
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("algo", [7, 8, 9, 10, 11, 101, 103])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_instantiation_matrix_two_bearers(width, algo, trace):
    c = Case(algo, CELLS[width], B=4, T=30, seed=31 * algo + 7 * trace + (width == "wide"), trace=trace, nb=2)
    g = c.scheduler()
    _check_width(g, width)
    bounds = [16, 30]
    c.check(c.run_host(g, bounds, 7), c.oracle(bounds))
    g.close()


# ---- 2. multi-TTI launches with finite queues, one bearer -------------------------------------------------------
@gpu
@pytest.mark.parametrize("refresh", [1, 40])
@pytest.mark.parametrize("algo", IDS)
def test_multi_tti_launches_with_queues(algo, refresh):
    """130 TTIs (64 does not divide it) in launches of 1, 7 and 64 TTIs: the kernel indexes every TTI's queues and
    delays while it keeps the cell state on chip."""
    c = Case(algo, CELLS["narrow"], B=5, T=130, seed=4000 + algo + refresh, queue=True, refresh=refresh)
    bounds = [80, 130]
    want = c.oracle(bounds)
    for tpl in (1, 7, 64):
        g = c.scheduler()
        c.check(c.run_host(g, bounds, tpl), want, tag=f"ttis_per_launch {tpl}")
        g.close()


# ---- 3. device-resident inputs ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("algo,nb", [(1, 1), (7, 1), (9, 1), (10, 1), (11, 1), (103, 1),
                                     (7, 2), (9, 2), (10, 2), (11, 2), (103, 2)])
def test_device_resident_queues(algo, nb, trace):
    """rs_run_device / rs_run_traces_device with queues, delays and the active mask in device memory (rs_set_queues
    with DEVICE pointers) == rs_run_host / rs_run_traces_host == the oracle."""
    c = Case(algo, CELLS["narrow"], B=5, T=30, seed=5000 + algo * 4 + nb * 2 + trace, trace=trace, queue=True, nb=nb)
    bounds = [14, 30]
    want = c.oracle(bounds)
    g = c.scheduler()
    c.check(c.run_host(g, bounds, 7), want, tag="host")
    g.reset_state()
    c.check(c.run_device(g, bounds, 7), want, tag="device")
    g.close()


# ---- 4. CQI staged in shared memory or read from global memory -------------------------------------------------
@gpu
@pytest.mark.parametrize("algo", [1, 7, 9, 103])
@pytest.mark.parametrize("layout", [0, 2])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_staging_on_and_off(width, layout, algo):
    """A handle under RS_NO_STAGE=1 reads every CQI from global memory; the default handle of a small batch stages
    it.  Streamed and trace-replayed CQI: the two are identical and equal the oracle."""
    for trace in (False, True):
        c = Case(algo, CELLS[width], B=4, T=20, seed=6000 + algo + 10 * layout + trace, layout=layout, trace=trace,
                 queue=trace)
        bounds = [9, 20]
        staged, plain = c.scheduler(), c.scheduler(RS_NO_STAGE=1)
        assert staged.smem_bytes > plain.smem_bytes
        a, b = c.run_host(staged, bounds, 7), c.run_host(plain, bounds, 7)
        _equal_runs(a, b, ("trace" if trace else "streamed"))
        c.check(a, c.oracle(bounds), tag="staged")
        staged.close()
        plain.close()


@gpu
def test_big_batch_refuses_staging_on_its_own():
    """BASELINE configs[3]'s 20 x 20 UE cell: a batch of 800 cells gives every SM more than the 4 staged cells that fit
    next to the CQI, so the library reads the CQI from global memory (same shared memory as an RS_NO_STAGE handle,
    less than a small batch's staged handle).  Device generators; the first and last cells against the oracle."""
    import torch
    S, n, B, T = 20, 20, 800, 6
    u2s = np.repeat(np.arange(S), n).astype(np.int32)
    U, G = len(u2s), 64
    w = 1.0 + (np.arange(S) % 3)
    w = w / w.sum()
    p = np.array([[0, 0, 1, 1] if s % 2 == 0 else [0, 0, 1, 0] for s in range(S)], dtype=np.int32)
    for layout in (0, 2):
        g = sched.Scheduler(9, w, p, u2s, B, cqi_per_rb=layout)
        with _env(RS_NO_STAGE=1):
            plain = sched.Scheduler(9, w, p, u2s, B, cqi_per_rb=layout)
        small = sched.Scheduler(9, w, p, u2s, 8, cqi_per_rb=layout)
        assert g.smem_bytes == plain.smem_bytes < small.smem_bytes, (g.smem_bytes, plain.smem_bytes, small.smem_bytes)
        plain.close()
        small.close()
        C = G // 2 if layout == 2 else G
        d_cqi = torch.empty((T, B, U, C), dtype=torch.uint8, device="cuda")
        d_r2 = torch.empty((T, B, 2), dtype=torch.int32, device="cuda")
        g.synth_cqi(3, 0, 0, T, d_cqi.data_ptr())
        g.synth_rand2(3, 0, 0, T, d_r2.data_ptr())
        d_out = {"rbg_to_ue": torch.empty((T, B, G), dtype=torch.int16, device="cuda"),
                 "tbs_bits": torch.empty((T, B, U), dtype=torch.int32, device="cuda"),
                 "mcs": torch.empty((T, B, U), dtype=torch.uint8, device="cuda"),
                 "final_cqi": torch.empty((T, B, U), dtype=torch.uint8, device="cuda"),
                 "slice_target": torch.empty((T, B, S), dtype=torch.int32, device="cuda"),
                 "slice_quota": torch.empty((T, B, S), dtype=torch.int32, device="cuda")}
        _, dts = workload.tti_clock(T)
        g.run_device(T, d_cqi.data_ptr(), B * U * C, d_r2.data_ptr(), dts, {k: v.data_ptr() for k, v in d_out.items()},
                     ttis_per_launch=4)
        g.sync()
        got = {k: v.cpu().numpy() for k, v in d_out.items()}
        st = g.get_state()
        cqi = workload.synth_cqi(3, 0, B, 0, T, U, G)
        r2 = d_r2.cpu().numpy()
        for sl in (slice(0, 4), slice(B - 4, B)):
            o = OracleScheduler(9, w, p, u2s, 4, n_threads=8)
            for t in range(T):
                want = o.step(cqi[t, sl], r2[t, sl], dt=float(dts[t]), want_aux=True)
                for k in got:
                    assert np.array_equal(want[k], got[k][t, sl]), (layout, t, k)
            so = o.get_state()
            for k in ("avg_rate", "tx_bytes", "cum_bytes", "cum_rbs", "slice_offset"):
                assert np.array_equal(so[k], st[k][sl]), (layout, k)
        g.close()


# ---- 5. part-batches ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("algo,nb", [(1, 1), (9, 1), (7, 2), (8, 2), (9, 2), (10, 2), (11, 2), (101, 2), (103, 2)])
def test_part_batches(algo, nb, trace):
    """RS_PARTS=3 on 7 cells (parts of 2, 2 and 3 cells, each launch offset by cell_off) with queues, delays and the
    active mask: identical to RS_PARTS=1 and equal to the oracle."""
    c = Case(algo, CELLS["narrow"], B=7, T=24, seed=7000 + algo * 4 + nb * 2 + trace, trace=trace, queue=True, nb=nb)
    bounds = [10, 24]
    parts, whole = c.scheduler(RS_PARTS=3), c.scheduler(RS_PARTS=1)
    a, b = c.run_host(parts, bounds, 5), c.run_host(whole, bounds, 5)
    _equal_runs(a, b, "parts")
    want = c.oracle(bounds)
    c.check(a, want)
    parts.reset_state()
    c.check(c.run_device(parts, bounds, 5), want, tag="device")
    parts.close()
    whole.close()


# ---- 6. cell widths: the LTE-Sim bands --------------------------------------------------------------------------
def _band_slices(n_rbs, rbg):
    """20 slices where there are fewer RBGs than that (quotas of 0 occur), else 7 uneven ones."""
    return [1, 2, 1, 1, 3, 1, 1, 2, 1, 1, 1, 2, 1, 1, 1, 1, 2, 1, 1, 1] if n_rbs // rbg < 8 else CELLS["narrow"]


@gpu
@pytest.mark.parametrize("algo", IDS)
@pytest.mark.parametrize("n_rbs,rbg", BANDS)
def test_lte_sim_bands(n_rbs, rbg, algo):
    """Every id on every band: layouts 0 and 1 (and the 4-bit layout where G % 8 == 0), backlogged and with finite
    queues, 20 TTIs in launches of 6."""
    G = n_rbs // rbg
    for layout in (0, 1, 2) if G % 8 == 0 else (0, 1):
        for queue in (False, True):
            c = Case(algo, _band_slices(n_rbs, rbg), B=4, T=20, seed=8000 + n_rbs + algo + 3 * layout + queue,
                     n_rbs=n_rbs, rbg=rbg, layout=layout, queue=queue)
            g = c.scheduler()
            bounds = [8, 20]
            c.check(c.run_host(g, bounds, 6), c.oracle(bounds), tag=(layout, queue))
            g.close()


@gpu
@pytest.mark.parametrize("i,band", list(enumerate(BANDS)))
def test_lte_sim_bands_trace_and_wide(i, band):
    """Per band one trace-replay case with queues and one 512-thread case, the ids rotating over the bands."""
    n_rbs, rbg = band
    G = n_rbs // rbg
    c = Case(IDS[i % 8], _band_slices(n_rbs, rbg), B=4, T=20, seed=9000 + i, n_rbs=n_rbs, rbg=rbg, trace=True, queue=True)
    g = c.scheduler()
    c.check(c.run_host(g, [7, 20], 6), c.oracle([7, 20]), tag="trace")
    g.close()
    c = Case(IDS[(i + 3) % 8], CELLS["wide"], B=3, T=12, seed=9100 + i, n_rbs=n_rbs, rbg=rbg, layout=2 if G % 8 == 0 else 0)
    g = c.scheduler()
    _check_width(g, "wide")
    c.check(c.run_host(g, [5, 12], 4), c.oracle([5, 12]), tag="wide")
    g.close()


# ---- 7. the widened fuzz -------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("seed", [1101, 1202, 1303])
def test_widened_fuzz(seed):
    """tools/fuzz_parity.one_case with the opt-in draws: LTE-Sim bands, two bearers, cells of up to ~600 UEs and the
    multi-TTI host / trace-replay entries with random launch lengths."""
    from tools import fuzz_parity
    rng = np.random.default_rng(seed)
    for case in range(4):
        err = fuzz_parity.one_case(rng, case, wide=True)
        assert err is None, f"seed {seed}: {err}"

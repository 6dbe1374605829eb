"""Per-slice buffer totals (rs_get_buffer_stats / rs_buffer_stats_device / rs_reduce_buffer_stats), tolerance 0: against
a numpy sum of the per-bearer buffers by slice and profile, and against the CPU buffer model of a closed loop."""
import ctypes as C

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.test_buffers_gpu import Traffic, buffered, host_run, oracle_loop
from tests.test_host_api_gpu import _nccl
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu


def summed(bufs, u2s, cell_profile, S):
    """uint64 [P][3][S] from rs_get_buffers' [B][U](nb) arrays: cell b adds to row cell_profile[b] with that profile's
    ue_to_slice (u2s [P][U])."""
    P = u2s.shape[0]
    out = np.zeros((P, 3, S), np.uint64)
    for b, p in enumerate(cell_profile):
        for k, key in enumerate(("queued", "dropped", "n_records")):
            per_ue = bufs[key][b].reshape(u2s.shape[1], -1).astype(np.uint64).sum(axis=1)
            np.add.at(out[p, k], u2s[p], per_ue)
    return out


def arrivals_run(g, c, u2s, cp, seed, K=6):
    """A closed loop of c.T TTIs through run_host with each profile's own arrival spec; slice 0 backlogged and, with two
    bearers, slot 0 of slice 3's UEs."""
    rng = np.random.default_rng(seed)
    P, S = u2s.shape[0], c.S
    pkt = rng.choice([0, 200, 1500], size=(P, S)).astype(np.int32)
    q16 = (rng.choice([0.2, 0.7, 3.5, 9.0], size=(P, S)) * 65536).astype(np.int32)
    pkt[:, 1], q16[:, 1] = 1500, 9 * 65536   # one slice overloaded: its FIFOs fill and drop
    arr = workload.synth_arrivals(seed, 0, c.B, 0, c.T, u2s, pkt, q16, n_bearers=c.nb, cell_profile=cp)
    s_of = u2s[cp]                           # [B][U]
    bl = np.repeat((s_of == 0)[..., None], c.nb, axis=2)
    if c.nb == 2:
        bl[..., 0] |= s_of == 3 % S
    g.enable_buffers(K, bl if c.nb == 2 else bl[..., 0])
    kw = dict(active=c.active, arrivals=arr, now=c.now, ttis_per_launch=16)
    if c.trace:
        g.run_traces_host(c.rows, c.draws, c.dts, **kw)
    else:
        g.run_host(c.slabs, c.draws, c.dts, **kw)


CASES = [(a, nb, P) for a in IDS for nb in (1, 2) for P in (1, 3) if not (a == 1 and nb == 2)]


@pytest.mark.parametrize("algo,nb,P", CASES)
def test_totals_equal_sum_of_buffers(algo, nb, P):
    c = Case(algo, CELLS["narrow"], B=7, T=40, seed=9100 + algo + 10 * nb + P, trace=algo % 2 == 1, nb=nb)
    if P == 1:
        g, u2s, cp = c.scheduler(), c.u2s[None], np.zeros(c.B, np.int64)
    else:
        u2s = np.stack([np.roll(c.u2s, 3 * p) for p in range(P)])
        cp = np.arange(c.B) % P
        g = sched.Scheduler.from_profiles(algo, [(c.w, c.p, m) for m in u2s], cp.astype(np.int32), **c.cfg())
        if c.trace:
            g.set_traces(c.traces, c.ue_trace)
    arrivals_run(g, c, u2s, cp, seed=algo + nb)
    bufs = g.get_buffers()
    want = summed(bufs, u2s, cp, c.S)
    got = g.get_buffer_stats()
    assert got.shape == ((3, c.S) if P == 1 else (P, 3, c.S))
    assert np.array_equal(got.reshape(P, 3, c.S), want)
    assert want[:, 0].sum() > 0 and want[:, 1].sum() > 0 and want[:, 2].sum() > 0   # queued, dropped and held
    g.close()


def test_totals_past_the_shared_memory_accumulators():
    """64 slices x 40 profiles: 3 x 64 x 40 sums are 60 KB, more than the 48 KB the kernel gathers in shared memory,
    so every bearer adds to global memory directly."""
    import torch
    S, P, B, T = 64, 40, 83, 24
    assert 3 * S * P * 8 > 48 * 1024
    rng = np.random.default_rng(3)
    base = np.repeat(np.arange(S), 2).astype(np.int32)
    u2s = np.stack([rng.permutation(base) for _ in range(P)])
    w = np.full(S, 1.0 / S)
    prm = np.tile(np.array([1, 1, 1, 1], np.int32), (S, 1))
    cp = (np.arange(B) * 7) % P
    g = sched.Scheduler.from_profiles(9, [(w, prm, m) for m in u2s], cp.astype(np.int32))
    U = u2s.shape[1]
    pkt = rng.choice([200, 1500], size=(P, S)).astype(np.int32)
    q16 = (rng.choice([0.3, 2.0, 6.0], size=(P, S)) * 65536).astype(np.int32)
    arr = workload.synth_arrivals(5, 0, B, 0, T, u2s, pkt, q16, cell_profile=cp)
    bl = rng.random((B, U)) < 0.2
    g.enable_buffers(5, bl)
    now, dts = workload.tti_clock(T)
    g.run_host(workload.synth_cqi(5, 0, B, 0, T, U, 64), workload.synth_rand2(5, 0, B, 0, T, S), dts, arrivals=arr,
               now=now, ttis_per_launch=8)
    want = summed(g.get_buffers(), u2s, cp, S)
    assert np.array_equal(g.get_buffer_stats(), want)
    assert want[:, 1].sum() > 0 and (want[:, 2] > 0).sum() > S
    d = torch.full((P * 3 * S,), 7, dtype=torch.int64, device="cuda")   # the device call clears its output first
    g.buffer_stats_device(d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64).reshape(P, 3, S), want)
    g.close()


@pytest.mark.parametrize("algo,nb,trace", [(9, 1, False), (10, 2, True), (7, 2, False), (103, 1, True)])
def test_closed_loop_totals_equal_cpu_model(algo, nb, trace):
    """120 TTIs of the device closed loop: the totals equal those of the CPU buffer model driving the oracle."""
    c = Case(algo, CELLS["narrow"], B=4, T=120, seed=9300 + algo + nb, trace=trace, nb=nb)
    tr = Traffic(c, seed=algo + 11 * nb)
    _, _, w_bufs = oracle_loop(c, tr, [120])
    g = buffered(c, tr)
    _, _, bufs = host_run(c, g, tr, [120], 16)
    for k in w_bufs[-1]:
        assert np.array_equal(bufs[-1][k], w_bufs[-1][k]), k
    want = summed(w_bufs[-1], c.u2s[None], np.zeros(c.B, np.int64), c.S)[0]
    assert np.array_equal(g.get_buffer_stats(), want)
    assert want[0].sum() > 0 and want[1].sum() > 0
    g.close()


def test_single_rank_reduce_equals_get():
    c = Case(9, CELLS["narrow"], B=6, T=40, seed=9400, nb=2)
    u2s = np.stack([c.u2s, np.roll(c.u2s, 5)])
    cp = np.arange(c.B) % 2
    g = sched.Scheduler.from_profiles(9, [(c.w, c.p, m) for m in u2s], cp.astype(np.int32), **c.cfg())
    arrivals_run(g, c, u2s, cp, seed=4)
    L = _nccl()
    L.rs_reduce_buffer_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    uid = (C.c_uint8 * 128)()
    assert L.rs_comm_unique_id(uid) == 0, L.rs_nccl_last_error()
    comm = C.c_void_p()
    assert L.rs_comm_init_rank(1, 0, uid, 0, C.byref(comm)) == 0, L.rs_nccl_last_error()
    red = np.zeros((2, 3, c.S), dtype=np.uint64)
    assert L.rs_reduce_buffer_stats(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, L.rs_nccl_last_error()
    L.rs_comm_destroy(comm)
    assert np.array_equal(red, g.get_buffer_stats()) and red[:, 0].sum() > 0
    g.close()


def test_unbuffered_handle_is_refused():
    import torch
    c = Case(9, CELLS["narrow"], B=2, T=1, seed=9500)
    g = c.scheduler()
    with pytest.raises(sched.RsError, match="rs_buffer_stats_device: the handle has no buffers"):
        g.get_buffer_stats()
    d = torch.zeros(3 * c.S, dtype=torch.int64, device="cuda")
    with pytest.raises(sched.RsError, match="no buffers"):
        g.buffer_stats_device(d.data_ptr())
    assert sched.lib().rs_buffer_stats_device(g._h, C.c_void_p(d.data_ptr())) == 1   # RS_ERR_ARG
    g.enable_buffers(4)
    assert np.array_equal(g.get_buffer_stats(), np.zeros((3, c.S), np.uint64))   # enabled, nothing arrived yet
    g.enable_buffers(0)
    with pytest.raises(sched.RsError, match="no buffers"):
        g.get_buffer_stats()
    g.close()


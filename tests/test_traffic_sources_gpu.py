"""GPU: traffic sources drawn on the device (rs_set_sources / rs_synth_traffic).  The generator equals its integer twin
workload.synth_traffic bit for bit; a buffered handle fed by it equals the CPU buffer model driving the oracle on the
twin's arrivals; rs_batch with periodic and on-off entries equals the Python mirror.  Tolerance 0 throughout."""
import os

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import SRC_NONE, SRC_ONOFF, SRC_PERIODIC, SRC_RATE
from tests import test_rs_batch_buffers_gpu as rbb
from tests.test_buffers_gpu import Traffic, assert_drains_and_builds, buffered, check, device_run, oracle_loop
from tests.helpers import ROOT
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu

ON, OFF = sched.onoff_spec(5, 8)
KINDS = [{"kind": SRC_NONE},
         {"kind": SRC_PERIODIC, "period_ttis": 5, "frame_bytes": [20000, 3000, 3000, 7000]},
         {"kind": SRC_ONOFF, "pkt_bytes": 700, "period_ttis": 2, "leave_on_q32": ON, "leave_off_q32": OFF},
         {"kind": SRC_RATE, "pkt_bytes": 200, "pkts_q16": sched.arrival_spec(200, 0.7)[1]}]


def _dev(shape):
    import torch
    return torch.zeros(shape, dtype=torch.int32, device="cuda")


def _profiles(S=4, U=7, P=3):
    rng = np.random.default_rng(P)
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([1, 1, 1, 1], np.int32), (S, 1))
    return [(w, p, rng.permutation(np.arange(U) % S).astype(np.int32)) for _ in range(P)]


@pytest.mark.parametrize("nb", [1, 2])
def test_device_equals_twin(nb):
    """Every kind, three profiles with their own rows, cells from 1000 on; one 64-TTI call, four 16-TTI calls after
    rs_set_sources again, and a 30-TTI call that continues the chains."""
    profs = _profiles()
    B, P = 37, 3
    cp = (np.arange(B) * 7 % P).astype(np.int32)
    rows = [KINDS, KINDS[::-1], [KINDS[2], KINDS[1], KINDS[2], KINDS[3]]]
    u2s = np.stack([m for _, _, m in profs])
    g = sched.Scheduler.from_profiles(9, profs, cp, n_bearers=nb)
    per = (B, 7, nb)
    want, st = workload.synth_traffic(77, 1000, B, 9, 94, u2s, rows, n_bearers=nb, cell_profile=cp)
    want = want.reshape((94,) + per)
    g.set_sources(rows)
    whole = _dev((64,) + per)
    g.synth_traffic(77, 1000, 9, 64, whole.data_ptr())
    g.set_sources(rows)                                   # restarts the chains: same draws again, in four calls
    parts = _dev((94,) + per)
    for k in range(4):
        g.synth_traffic(77, 1000, 9 + 16 * k, 16, parts[16 * k].data_ptr())
    g.synth_traffic(77, 1000, 73, 30, parts[64].data_ptr())
    g.sync()
    assert np.array_equal(whole.cpu().numpy(), want[:64])
    assert np.array_equal(parts.cpu().numpy(), want)
    assert {int(x) for x in np.unique(want)} >= {0, 700, 20000, 3000, 7000, 200}


def test_argument_checks_and_restart():
    profs = _profiles(P=1)
    w, p, u2s = profs[0]
    g = sched.Scheduler(9, w, p, u2s, 6, n_bearers=2)
    d = _dev((40, 6, 7, 2))
    with pytest.raises(sched.RsError, match="no sources"):
        g.synth_traffic(1, 0, 0, 8, d.data_ptr())
    g.set_sources(KINDS)
    g.synth_traffic(1, 4, 3, 8, d.data_ptr())
    for seed, cell0, tti0, what in [(1, 4, 12, "continue at tti0 11"), (1, 4, 10, "tti0 11"), (2, 4, 11, "seed 1"),
                                    (1, 5, 11, "cell0 4"), (1, 4, -1, "bad argument")]:
        with pytest.raises(sched.RsError, match=what):
            g.synth_traffic(seed, cell0, tti0, 8, d.data_ptr())
    bad = [(dict(KINDS[0], kind=7), "kind 7"), (dict(KINDS[1], period_ttis=0), "period_ttis 0"),
           (dict(KINDS[1], frame_bytes=[]), "n_frames 0"), (dict(KINDS[1], frame_bytes=[5, 0]), r"frame_bytes\[1\] = 0"),
           (dict(KINDS[1], frame_bytes=[1] * 1025), "n_frames 1025"), (dict(KINDS[2], pkt_bytes=0), "pkt_bytes 0"),
           (dict(KINDS[2], leave_off_q32=0), "a leaving probability of 0"),
           (dict(KINDS[3], pkt_bytes=10 ** 9, pkts_q16=3 * 65536), "a TTI's bytes overflow int32"),
           (dict(KINDS[3], pkts_q16=-1), "negative")]
    for e, what in bad:
        src = list(KINDS)
        src[2] = e
        with pytest.raises(sched.RsError, match=f"rs error 1: rs_set_sources: profile 0 slice 2: {what}"):
            g.set_sources(src)
    # nothing was half-applied, and rs_synth_arrivals (its own table) leaves the sources alone: the chains continue
    g.synth_arrivals(1, 4, 11, 8, np.full((1, 4), 100), np.full((1, 4), 65536), d[20].data_ptr())
    g.synth_traffic(1, 4, 11, 8, d[8].data_ptr())
    g.sync()
    want, st = workload.synth_traffic(1, 4, 6, 3, 16, u2s, KINDS, n_bearers=2)
    assert np.array_equal(d[:16].cpu().numpy(), want)
    assert np.array_equal(d[20:28].cpu().numpy(), np.full((8, 6, 7, 2), 100))
    # rs_set_sources again restarts the chains at any tti0
    g.set_sources(KINDS)
    g.synth_traffic(1, 4, 500, 20, d.data_ptr())
    g.sync()
    again, _ = workload.synth_traffic(1, 4, 6, 500, 20, u2s, KINDS, n_bearers=2)
    assert np.array_equal(d[:20].cpu().numpy(), again)
    g.close()


class SourceTraffic(Traffic):
    """test_buffers_gpu's Traffic (backlogged bearers, clock) with arrivals from the sources: slice 0 none, then periodic
    frames that overload their bearers, on-off packets and a rate that drain, in turn."""

    def __init__(self, c, seed):
        super().__init__(c, seed)
        self.sources = [KINDS[0]] + [KINDS[1 + (s - 1) % 3] for s in range(1, c.S)]
        self.arr, _ = workload.synth_traffic(seed, 0, c.B, 0, c.T, c.u2s, self.sources, n_bearers=c.nb)


class _DrawsSources:
    """The handle as test_buffers_gpu.device_run uses it, with its arrivals drawn by rs_synth_traffic."""

    def __init__(self, g, sources):
        self._g = g
        g.set_sources(sources)

    def __getattr__(self, name):
        return getattr(self._g, name)

    def synth_arrivals(self, seed, cell0, tti0, n_ttis, pkt_bytes, pkts_q16, d_out):
        self._g.synth_traffic(seed, cell0, tti0, n_ttis, d_out)


@pytest.mark.parametrize("algo", IDS)
def test_closed_loop_on_device_sources_matches_oracle(algo):
    """Schedules, state, queue_out / hol_out and the buffers at each call boundary of a buffered handle fed by
    rs_synth_traffic, against tests/buffer_model.py + the oracle fed by the twin's arrivals."""
    nb = 1 if algo == 1 else 2
    c = Case(algo, CELLS["narrow"], B=5, T=70, seed=8100 + algo, nb=nb)
    tr = SourceTraffic(c, seed=40 + algo)
    bounds = [33, 70]
    want = oracle_loop(c, tr, bounds)
    assert_drains_and_builds(want[0], tr)
    g = buffered(c, tr)
    check(c, device_run(c, _DrawsSources(g, tr.sources), tr, bounds, 7), want, tag="device sources")
    g.close()


# ---- rs_batch --traffic with every entry form ------------------------------------------------------------------------
GROUPS4 = [(1, 0.3, (0, 0, 1, 1)), (1, 0.2, (1, 1, 1, 1)), (1, 0.2, (1, 1, 1, 1)), (2, 0.3, (1, 0, 1, 0))]
MIXED = [{"backlogged": 1}, {"period_ttis": 4, "frame_bytes": [9000, 1500, 1500]},
         {"pkt_bytes": 900, "period_ttis": 3, "on_ttis": 6, "off_ttis": 9}, {"pkt_bytes": 1500, "pkts_per_tti": 9}]


class _Delegate:
    def __init__(self, mod, **override):
        self._mod = mod
        self.__dict__.update(override)

    def __getattr__(self, name):
        return getattr(self._mod, name)


@pytest.fixture
def mirror(monkeypatch):
    """test_rs_batch_buffers_gpu.mirror with the traffic read by sched.load_traffic and drawn by workload.synth_traffic."""
    monkeypatch.setattr(rbb, "sched", _Delegate(sched, load_traffic_config=lambda t, c: sched.load_traffic(t, c) + (None,)))
    monkeypatch.setattr(rbb, "workload", _Delegate(workload, synth_arrivals=lambda seed, c0, B, t0, T, u2s, src, _, n_bearers,
                                                   cell_profile: workload.synth_traffic(
                                                       seed, c0, B, t0, T, u2s, [list(r) for r in src], n_bearers=n_bearers,
                                                       cell_profile=cell_profile)[0]))
    return rbb.mirror


def _files(tmp_path, nb, P):
    out = []
    for p in range(P):
        groups = GROUPS4 if p == 0 else [(n, w, (a, b, 1 - e, s)) for n, w, (a, b, e, s) in GROUPS4[::-1]]
        out.append(rbb._files(tmp_path, nb, tag=str(p), groups=groups, traffic=MIXED if p == 0 else MIXED[::-1]))
    return out


@pytest.mark.parametrize("algo,replay,nb,P", [(9, False, 1, 1), (9, True, 2, 2), (8, False, 2, 1), (7, False, 1, 2),
                                              (10, False, 2, 1), (103, True, 1, 1), (11, False, 2, 1)])
def test_rs_batch_sources_equal_python_mirror(algo, replay, nb, P, tmp_path, mirror):
    B, T, seed, log_cell = 19, 45, 6, 7
    cfgs, trafs = zip(*_files(tmp_path, nb, P))
    args = ["--algo", algo, "--cells", B, "--ttis", T, "--seed", seed, "--buffers", rbb.K, "--log-cell", log_cell,
            "--log-prefix", tmp_path / "cell"]
    for c, t in zip(cfgs, trafs):
        args += ["--config", c, "--traffic", t]
    rep = None
    if replay:
        targs, traces, mp, n_rows = rbb._traces(tmp_path)
        args += targs
        rep = (traces, mp, n_rows)
    lines = rbb._run(*args)
    st, bs, out, err = mirror(algo, cfgs, trafs, B, T, seed, log_cell, rep)
    rbb.check_lines(lines, st, bs, B, P)
    assert (tmp_path / "cell.stdout").read_text() == out
    assert (tmp_path / "cell.stderr").read_text() == err
    assert err.count("\n") > T


def test_rs_batch_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 is compared with --gpus 1 only where two are present")
    (cfg, traffic), = _files(tmp_path, 2, 1)
    runs = []
    for n in (1, 2):
        runs.append(rbb._run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", rbb.K, "--cells", 301, "--ttis",
                             64, "--seed", 3, "--gpus", n, "--log-cell", 200, "--log-prefix", tmp_path / f"c{n}")[0])
    for k in ("slice_bytes", "slice_rbs", "queued_bytes", "dropped_bytes", "records"):
        assert runs[0][k] == runs[1][k], k
    for ext in ("stdout", "stderr"):
        assert (tmp_path / f"c1.{ext}").read_text() == (tmp_path / f"c2.{ext}").read_text()


def test_shipped_example_runs(tmp_path, mirror):
    """rs_batch on cfg20x5_ab.json with tests/data/traffic20x5_video_voip.json equals the mirror."""
    d = os.path.join(ROOT, "tests", "data")
    cfg, traffic = os.path.join(d, "cfg20x5_ab.json"), os.path.join(d, "traffic20x5_video_voip.json")
    lines = rbb._run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", rbb.K, "--cells", 16, "--ttis", 300,
                     "--seed", 2)
    st, bs, _, _ = mirror(9, [cfg], [traffic], 16, 300, 2, 0)
    assert lines[0]["slice_bytes"] == [int(x) for x in st[0, 0]] and lines[0]["slice_rbs"] == [int(x) for x in st[0, 1]]
    for k, name in enumerate(("queued_bytes", "dropped_bytes", "records")):
        assert lines[0][name] == [int(x) for x in bs[0, k]]
    assert sum(lines[0]["records"]) > 0

"""GPU: the synthetic channel drawn on the device (rs_set_channels / rs_synth_channel).  The generator equals its integer
twin workload.synth_channel bit for bit; fading CQI it draws, fed to rs_run_device with cqi_refresh 40, schedules what
the CPU oracle schedules on the twin's CQI; rs_batch --channel equals the Python mirror.  Tolerance 0 throughout."""
import json
import os

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import CH_IID
from tests import test_rs_batch_buffers_gpu as rbb
from tests.helpers import ROOT
from tests.test_kernel_paths_gpu import CELLS, IDS, Case

pytestmark = pytest.mark.gpu

COUNTS = [0, 0, 1, 2, 5, 9, 14, 20, 25, 20, 14, 9, 5, 2, 0]
IID = {"kind": CH_IID}
FADE = sched.channel_spec(COUNTS, 1.5, 6, 4)
EDGE = sched.channel_spec([30, 40, 20, 10] + [0] * 11, 2.5, 1, 1)         # low levels, clamped at 1, white offsets
FLAT = sched.channel_spec(COUNTS[::-1], 0.75, 0, 0)                        # flat and frozen


def _dev(shape):
    import torch
    return torch.zeros(shape, dtype=torch.uint8, device="cuda")


def _profiles(S=4, U=9, P=3):
    rng = np.random.default_rng(P)
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([0, 0, 1, 1], np.int32), (S, 1))
    return [(w, p, rng.permutation(np.arange(U) % S).astype(np.int32)) for _ in range(P)]


def _layout(cqi, layout):
    return sched.pack_cqi(cqi) if layout == 2 else cqi


@pytest.mark.parametrize("layout", [0, 2])
@pytest.mark.parametrize("P", [1, 3])
def test_device_equals_twin(layout, P):
    """Mixed IID / FADING slices, one profile or three with their own rows, cells from 1000 and epochs from 37 on; one
    12-slab call and the same epochs in calls of 5 and 7 slabs."""
    profs = _profiles(P=P)
    B = 29
    rows = [[FADE, IID, EDGE, FLAT], [IID, FLAT, FADE, EDGE], [EDGE, FADE, IID, IID]][:P]
    u2s = np.stack([m for _, _, m in profs])
    if P == 1:
        cp = None
        g = sched.Scheduler(9, *profs[0], B, cqi_per_rb=layout)
    else:
        cp = (np.arange(B) * 7 % P).astype(np.int32)
        g = sched.Scheduler.from_profiles(9, profs, cp, cqi_per_rb=layout)
    want = _layout(workload.synth_channel(77, 1000, B, 37, 12, u2s, rows, cell_profile=cp), layout)
    g.set_channels(rows if P > 1 else rows[0])
    whole, parts = _dev(want.shape), _dev(want.shape)
    g.synth_channel(77, 1000, 37, 12, whole.data_ptr())
    g.synth_channel(77, 1000, 37, 5, parts.data_ptr())
    g.synth_channel(77, 1000, 42, 7, parts[5].data_ptr())
    g.sync()
    assert np.array_equal(whole.cpu().numpy(), want)
    assert np.array_equal(parts.cpu().numpy(), want)
    full = workload.synth_channel(77, 1000, B, 37, 12, u2s, rows, cell_profile=cp)
    assert len(np.unique(full)) >= 12
    g.close()


@pytest.mark.parametrize("n_rbs,rbg,layout", [(100, 4, 0), (48, 3, 0), (384, 8, 2), (64, 8, 2)])
def test_device_equals_twin_below_64_rbgs(n_rbs, rbg, layout):
    """G = 25 and 16 RBGs in layout 0 (lanes past G store nothing), G = 48 and 8 in layout 2 (G / 2 lanes store a row's
    bytes, the upper half from RBGs 32..): rows narrower than the warp's 64 RBGs land in the handle's row width."""
    G = n_rbs // rbg
    w, p, u2s = _profiles(P=1)[0]
    g = sched.Scheduler(9, w, p, u2s, 11, n_rbs=n_rbs, rbg_size=rbg, cqi_per_rb=layout)
    rows = [FADE, IID, EDGE, FLAT]
    g.set_channels(rows)
    want = _layout(workload.synth_channel(21, 40, 11, 5, 3, u2s, rows, n_rbgs=G), layout)
    assert want.shape[-1] == g.cqi_cols
    d = _dev(want.shape)
    g.synth_channel(21, 40, 5, 3, d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy(), want)
    g.close()


def test_more_than_4096_ues():
    """U = 4100: UEs u and u + 4096 share the low 12 bits of the counter (the ue >> 12 fold keeps them apart)."""
    U = 4100
    u2s = (np.arange(U) % 2).astype(np.int32)
    g = None
    for algo in (1, 8, 9):   # the first id whose cell of 4100 UEs fits one CTA
        try:
            g = sched.Scheduler(algo, np.full(2, 0.5), np.ones((2, 4), np.int32), u2s, 3, cqi_per_rb=2)
            break
        except sched.RsError:
            continue
    assert g is not None, "no id takes a cell of 4100 UEs"
    g.set_channels([FADE, IID])
    want = sched.pack_cqi(workload.synth_channel(5, 7, 3, 2, 3, u2s, [FADE, IID]))
    d = _dev(want.shape)
    g.synth_channel(5, 7, 2, 3, d.data_ptr())
    g.sync()
    assert np.array_equal(d.cpu().numpy(), want)
    assert not np.array_equal(want[:, :, 2], want[:, :, 4098]) and not np.array_equal(want[:, :, 3], want[:, :, 4099])
    g.close()


@pytest.mark.parametrize("layout", [0, 2])
def test_all_iid_equals_synth_cqi(layout):
    w, p, u2s = _profiles(P=1)[0]
    g = sched.Scheduler(9, w, p, u2s, 40, cqi_per_rb=layout)
    g.set_channels([IID] * 4)
    shape = (9, 40, 9, 64 if layout == 0 else 32)
    a, b = _dev(shape), _dev(shape)
    g.synth_channel(3, 500, 81, 9, a.data_ptr())
    g.synth_cqi(3, 500, 81, 9, b.data_ptr())
    g.sync()
    assert np.array_equal(a.cpu().numpy(), b.cpu().numpy())
    g.close()


def test_argument_checks():
    w, p, u2s = _profiles(P=1)[0]
    g = sched.Scheduler(9, w, p, u2s, 6, cqi_per_rb=2)
    d = _dev((2, 4, 6, 9, 32))
    with pytest.raises(sched.RsError, match="rs error 1: rs_synth_channel: no channels"):
        g.synth_channel(1, 0, 0, 2, d.data_ptr())
    rows = [FADE, IID, EDGE, FLAT]
    g.set_channels(rows)
    g.synth_channel(1, 3, 10, 4, d[0].data_ptr())
    bad = [(dict(FADE, kind=5), "kind 5 is not RS_CH_IID or RS_CH_FADING"), (dict(FADE, depth_q8=3841), "depth_q8 3841"),
           (dict(FADE, depth_q8=-1), "depth_q8 -1"), (dict(FADE, coherence_rbgs=-1), "coherence_rbgs -1 is below 0"),
           (dict(FADE, coherence_epochs=-3), "coherence_epochs -3 is below 0"),
           (dict(FADE, level_thr=[5] * 7 + [4] * 7), r"level_thr\[7\] < level_thr\[6\]")]
    for e, what in bad:
        with pytest.raises(sched.RsError, match=f"rs error 1: rs_set_channels: profile 0 slice 2: {what}"):
            g.set_channels([FADE, IID, e, FLAT])
    # the refused calls changed nothing: the next draw equals the one made before them
    g.synth_channel(1, 3, 10, 4, d[1].data_ptr())
    g.sync()
    assert np.array_equal(d[0].cpu().numpy(), d[1].cpu().numpy())
    assert np.array_equal(d[0].cpu().numpy(), sched.pack_cqi(workload.synth_channel(1, 3, 6, 10, 4, u2s, rows)))
    g.close()
    per_rb = sched.Scheduler(9, w, p, u2s, 6, cqi_per_rb=1)
    per_rb.set_channels(rows)
    with pytest.raises(sched.RsError, match="rs error 2: synthetic CQI is one value per RBG"):
        per_rb.synth_channel(1, 0, 0, 1, d.data_ptr())
    per_rb.close()


@pytest.mark.parametrize("algo", IDS)
def test_device_fading_cqi_schedules_like_the_oracle(algo):
    """Slabs drawn by rs_synth_channel in the packed layout, read every 40 TTIs by rs_run_device, against the oracle fed
    the twin's CQI: every output of every TTI and the state at each call boundary."""
    c = Case(algo, CELLS["narrow"], B=6, T=100, seed=9300 + algo, layout=2, refresh=40)
    rows = [FADE, EDGE, IID, FLAT, FADE, EDGE, FLAT]
    g = c.scheduler()
    g.set_channels(rows)
    slabs = workload.synth_channel(c.B + algo, 0, c.B, 0, 3, c.u2s, rows)
    c.ocqi = slabs[np.arange(c.T) // 40]
    d = _dev((3, c.B, c.U, c.G // 2))
    g.synth_channel(c.B + algo, 0, 0, 3, d.data_ptr())
    g.sync()
    c.slabs = d.cpu().numpy()
    assert np.array_equal(c.slabs, sched.pack_cqi(slabs))
    bounds = [40, 100]
    c.check(c.run_device(g, bounds, 16), c.oracle(bounds), tag="device channel")
    g.close()


# ---- rs_batch --channel ----------------------------------------------------------------------------------------------
GROUPS = [(3, 0.2, (0, 0, 1, 1)), (2, 0.2, (0, 0, 1, 0))]
UES = [4, 2, 6, 1, 3]
SPEC = {"level_counts": COUNTS, "depth_cqi": 1.5, "coherence_rbgs": 6, "coherence_reports": 4}
EDGE_SPEC = {"level_counts": [30, 40, 20, 10] + [0] * 11, "depth_cqi": 2.5, "coherence_rbgs": 1, "coherence_reports": 1}


def _config(tmp_path, tag="", groups=GROUPS):
    cfg = {"slices": [{"n_slices": n, "weight": w, "algo_alpha": a, "algo_beta": b, "algo_epsilon": e, "algo_psi": p}
                      for n, w, (a, b, e, p) in groups], "ues_per_slice": UES}
    path = tmp_path / f"cfg{tag}.json"
    path.write_text(json.dumps(cfg))
    return str(path)


def _channel_file(tmp_path, entries, report, tag=""):
    path = tmp_path / f"channel{tag}.json"
    path.write_text(json.dumps({"report_ttis": report, "slices": entries, "note": "test"}))
    return str(path)


def _channel_cqi(cfgs, chans, B, T, seed):
    """uint8 [T][B][U][64]: the CQI each TTI of rs_batch --channel reads (report e = epoch e, at TTIs e * R ..)."""
    loaded = [sched.load_channel(f, c) for c, f in zip(cfgs, chans)]
    rep = loaded[0][0]
    P = len(cfgs)
    u2s = np.stack([sched.load_slice_config(c)[2] for c in cfgs])
    slabs = workload.synth_channel(seed, 0, B, 0, (T - 1) // rep + 1, u2s, [ch for _, ch in loaded],
                                   cell_profile=np.arange(B) % P)
    return slabs[np.arange(T) // rep]


def _mirror(algo, cfg, B, T, seed, log_cell, cqi):
    """rs_batch without buffers through the ctypes mirror: (slice totals, log stdout, stderr)."""
    w, p, u2s = sched.load_slice_config(cfg)
    S = len(w)
    g = sched.Scheduler(algo, w, p, u2s, B, cqi_per_rb=2)
    draws = workload.synth_rand2(seed, 0, B, 0, T, S)
    _, dts = workload.tti_clock(T)
    res = g.run_host(sched.pack_cqi(cqi), draws, dts, want_aux=True, ttis_per_launch=16)
    st = g.get_stats()
    g.close()
    lw = sched.LogWriter(algo, u2s, S, cqi_per_rb=2)
    c = log_cell
    for t in range(T):
        lw.tti(100 + t, sched.pack_cqi(cqi[t, c]), res["rbg_to_ue"][t, c], res["tbs_bits"][t, c], res["final_cqi"][t, c],
               res["slice_target"][t, c], res["slice_quota"][t, c])
    return st, lw.stdout, lw.stderr


@pytest.mark.parametrize("report", [1, 7, 40])
def test_rs_batch_channel_equals_python_mirror(report, tmp_path):
    """Reports every 1, 7 (divides no chunk of 16) and 40 TTIs over 95 TTIs: chunks that cross a report still read its
    slab, and --log-cell logs the CQI each TTI used."""
    B, T, seed, log_cell = 37, 95, 4, 11
    cfg = _config(tmp_path)
    ch = _channel_file(tmp_path, [SPEC, {"iid": 1}], report)
    got = rbb._run("--algo", 9, "--config", cfg, "--channel", ch, "--cells", B, "--ttis", T, "--seed", seed,
                   "--log-cell", log_cell, "--log-prefix", tmp_path / "cell")[0]
    cqi = _channel_cqi([cfg], [ch], B, T, seed)
    st, out, err = _mirror(9, cfg, B, T, seed, log_cell, cqi)
    assert got["slice_bytes"] == [int(x) for x in st[0]] and got["slice_rbs"] == [int(x) for x in st[1]]
    assert got["cqi"] == "synthetic" and got["cells"] == B and got["ttis"] == T
    assert (tmp_path / "cell.stdout").read_text() == out
    assert (tmp_path / "cell.stderr").read_text() == err
    assert err.count("\n") > T


@pytest.mark.parametrize("algo,nb,report", [(9, 1, 7), (8, 2, 40), (10, 2, 1)])
def test_rs_batch_channel_with_buffers_equals_python_mirror(algo, nb, report, tmp_path, monkeypatch):
    """--buffers --traffic with a channel file per config (two configs): test_rs_batch_buffers_gpu's mirror with the
    channel's CQI in place of synth_cqi."""
    B, T, seed, log_cell = 19, 45, 6, 7
    cfgs, trafs = zip(*[rbb._files(tmp_path, nb, tag=str(p),
                                   groups=rbb.GROUPS if p == 0 else [(n, w, (a, b, 1 - e, s)) for n, w, (a, b, e, s) in rbb.GROUPS[::-1]],
                                   traffic=rbb.TRAFFIC if p == 0 else rbb.TRAFFIC[::-1]) for p in range(2)])
    chans = [_channel_file(tmp_path, [SPEC, EDGE_SPEC, {"iid": 1}], report, tag="0"),
             _channel_file(tmp_path, [{"iid": 1}, SPEC, EDGE_SPEC], report, tag="1")]
    args = ["--algo", algo, "--cells", B, "--ttis", T, "--seed", seed, "--buffers", rbb.K, "--log-cell", log_cell,
            "--log-prefix", tmp_path / "cell"]
    for c, t, h in zip(cfgs, trafs, chans):
        args += ["--config", c, "--traffic", t, "--channel", h]
    lines = rbb._run(*args)
    cqi = _channel_cqi(cfgs, chans, B, T, seed)

    class _W:
        def __getattr__(self, name):
            return getattr(workload, name)

        @staticmethod
        def synth_cqi(*_):
            return cqi

    monkeypatch.setattr(rbb, "workload", _W())
    st, bs, out, err = rbb.mirror(algo, cfgs, trafs, B, T, seed, log_cell)
    rbb.check_lines(lines, st, bs, B, 2)
    assert (tmp_path / "cell.stdout").read_text() == out
    assert (tmp_path / "cell.stderr").read_text() == err


def _without_rate(line):
    return {k: v for k, v in line.items() if k != "cell_ttis_per_s"}


def test_rs_batch_all_iid_file_equals_no_flag(tmp_path):
    """A file of {"iid": 1} entries with report_ttis 1 gives the output of the run without --channel: the same lines
    (but the measured rate) and the same log text, byte for byte."""
    cfg = _config(tmp_path)
    ch = _channel_file(tmp_path, [{"iid": 1}] * 2, 1)
    runs = []
    for extra, tag in (([], "plain"), (["--channel", ch], "iid")):
        runs.append(rbb._run("--algo", 9, "--config", cfg, "--cells", 53, "--ttis", 70, "--seed", 8, "--log-cell", 30,
                             "--log-prefix", tmp_path / tag, *extra))
    assert [_without_rate(x) for x in runs[0]] == [_without_rate(x) for x in runs[1]]
    for ext in ("stdout", "stderr"):
        assert (tmp_path / f"plain.{ext}").read_bytes() == (tmp_path / f"iid.{ext}").read_bytes()


def test_rs_batch_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 --channel is compared with --gpus 1 only where two are present")
    cfg = _config(tmp_path)
    ch = _channel_file(tmp_path, [SPEC, EDGE_SPEC], 7)
    runs = []
    for n in (1, 2):
        runs.append(rbb._run("--algo", 9, "--config", cfg, "--channel", ch, "--cells", 301, "--ttis", 64, "--seed", 3,
                             "--gpus", n, "--log-cell", 200, "--log-prefix", tmp_path / f"c{n}")[0])
    for k in ("slice_bytes", "slice_rbs"):
        assert runs[0][k] == runs[1][k], k
    for ext in ("stdout", "stderr"):   # cell 200 lives on GPU 1
        assert (tmp_path / f"c1.{ext}").read_text() == (tmp_path / f"c2.{ext}").read_text()


def test_shipped_example_runs(tmp_path):
    """rs_batch on cfg20x5.json with tests/data/channel20x5_traces.json (reports every 40 TTIs) equals the mirror."""
    d = os.path.join(ROOT, "tests", "data")
    cfg, ch = os.path.join(d, "cfg20x5.json"), os.path.join(d, "channel20x5_traces.json")
    B, T = 16, 130
    got = rbb._run("--algo", 9, "--config", cfg, "--channel", ch, "--cells", B, "--ttis", T, "--seed", 2,
                   "--log-cell", 3, "--log-prefix", tmp_path / "cell")[0]
    st, _, err = _mirror(9, cfg, B, T, 2, 3, _channel_cqi([cfg], [ch], B, T, 2))
    assert got["slice_bytes"] == [int(x) for x in st[0]] and got["slice_rbs"] == [int(x) for x in st[1]]
    assert (tmp_path / "cell.stderr").read_text() == err

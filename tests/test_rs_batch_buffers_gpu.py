"""GPU: rs_batch --buffers K --traffic FILE, the closed loop of the C++ batch program.  Its per-slice throughput and
buffer totals and its --log-cell text must equal the same run through the Python mirror (Scheduler + enable_buffers +
workload.synth_arrivals, traffic read by load_traffic_config) on the same seeds and the same clock, tolerance 0."""
import json
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

pytestmark = pytest.mark.gpu
BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
FIX = os.path.join(ROOT, "tests", "golden", "traces", "trace_subset.npz")
K = 6
G = 64
# slice groups: backlogged PF; alpha/beta slices weighted by delay; an alpha-only slice
GROUPS = [(1, 0.3, (0, 0, 1, 1)), (2, 0.3, (1, 1, 1, 1)), (2, 0.4, (1, 0, 1, 0))]
UES = [3, 2, 4, 1, 3]
TRAFFIC = [{"backlogged": 1}, {"pkt_bytes": 1500, "pkts_per_tti": 9}, {"pkt_bytes": 300, "pkts_per_tti": 2.5}]


def _files(tmp_path, nb, tag="", groups=GROUPS, traffic=TRAFFIC):
    cfg = {"slices": [{"n_slices": n, "weight": w, "algo_alpha": a, "algo_beta": b, "algo_epsilon": e, "algo_psi": p,
                       "internet_flow": 2, "if_bitrate": [9, 3]}       # read by neither side
                      for n, w, (a, b, e, p) in groups], "ues_per_slice": UES}
    c, t = tmp_path / f"cfg{tag}.json", tmp_path / f"traffic{tag}.json"
    c.write_text(json.dumps(cfg, indent=1))
    t.write_text(json.dumps({"bearers": nb, "slices": traffic}))
    return str(c), str(t)


def _run(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    r = subprocess.run([BIN, *[str(a) for a in args]], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    return [json.loads(x) for x in r.stdout.strip().splitlines()]


def _traces(tmp_path):
    """The trace fixture as ue<id>.log files + a mapping file, and the arrays rs_batch reads from them."""
    z = np.load(FIX)
    ids, rows = z["trace_ids"], z["rows"]
    n_rows = rows.shape[1]
    tdir = tmp_path / "traces"
    tdir.mkdir()
    for k in range(6):
        per_rb = np.repeat(rows[k], 8, axis=1)
        (tdir / f"ue{int(ids[k])}.log").write_text("\n".join(" ".join(str(int(v)) for v in r) for r in per_rb) + "\n")
    mp = ids[np.random.default_rng(2).integers(0, 6, 23)]
    (tmp_path / "mapping.config").write_text("".join(f"{i} {int(t)}\n" for i, t in enumerate(mp)))
    traces = np.full((int(mp.max()) + 1, n_rows, 512), 10, dtype=np.uint8)
    for k in range(6):
        traces[int(ids[k])] = np.repeat(rows[k], 8, axis=1)
    args = ["--traces", tdir, "--mapping", tmp_path / "mapping.config", "--trace-rows", n_rows]
    return args, traces, mp, n_rows


def mirror(algo, cfgs, trafs, B, T, seed, log_cell, replay=None):
    """The same closed loop through the ctypes mirror: ({slice totals, buffer totals} per config, log stdout, stderr)."""
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
    if algo == 10:
        g.set_grant_list_len(max(S * G, 2 * G))   # as the program does for its logged cell
    g.enable_buffers(K, np.stack([tr[c][1] for c in cp]))
    all_u2s = np.stack([pr[2] for pr in profs])
    arr = workload.synth_arrivals(seed, 0, B, 0, T, all_u2s, np.stack([t[2] for t in tr]), np.stack([t[3] for t in tr]),
                                  n_bearers=nb, cell_profile=cp)
    now, dts = workload.tti_clock(T)
    if algo == 11:
        draws = workload.synth_rand_draws(seed, 0, B, 0, T, S, g.rand_stride)
    else:
        draws = workload.synth_rand2(seed, 0, B, 0, T, S)
    kw = dict(want_aux=True, ttis_per_launch=16, arrivals=arr, now=now)
    if replay is None:
        cqi = workload.synth_cqi(seed, 0, B, 0, T, U, G)
        res = g.run_host(sched.pack_cqi(cqi), draws, dts, **kw)
        cqi_of = lambda t: sched.pack_cqi(cqi[t, log_cell])   # noqa: E731
    else:
        traces, mp, n_rows = replay
        ue_trace = np.array([[mp[(u + 7 * b) % len(mp)] for u in range(U)] for b in range(B)], dtype=np.int32)
        g.set_traces(traces, ue_trace)
        rows = sched.trace_rows_for_run(now, 0, n_rows=n_rows)
        res = g.run_traces_host(rows, draws, dts, **kw)
        cqi_of = lambda t: sched.pack_cqi(np.stack([traces[ue_trace[log_cell, u], rows[t], ::8] if rows[t] >= 0   # noqa: E731
                                                    else np.full(G, 10, np.uint8) for u in range(U)]))
    st, bs = g.get_stats().reshape(P, 4, S), g.get_buffer_stats().reshape(P, 3, S)
    g.close()
    lp = log_cell % P
    lw = sched.LogWriter(algo, profs[lp][2], S, cqi_per_rb=2, n_bearers=nb)
    c = log_cell
    for t in range(T):
        q, h = res["queue_out"][t, c], res["hol_out"][t, c]
        if algo == 10:
            lw.tti_grants(100 + t, cqi_of(t), int(res["alloc_n"][t, c]), res["alloc_ue"][t, c], res["alloc_rbg"][t, c],
                          res["tbs_bits"][t, c], res["final_cqi"][t, c], res["slice_target"][t, c],
                          res["slice_quota"][t, c], queue=q, hol=h)
            continue
        transport = algo in (8, 9, 101, 103)
        lw.tti(100 + t, cqi_of(t), res["rbg_to_ue"][t, c], res["tbs_bits"][t, c],
               res["final_cqi"][t, c] if algo != 1 else None, res["slice_target"][t, c] if transport else None,
               res["slice_quota"][t, c] if transport else None, queue=q, hol=h)
    return st, bs, lw.stdout, lw.stderr


def check_lines(lines, st, bs, B, P):
    assert len(lines) == P
    for p, got in enumerate(lines):
        assert got["cells"] == B // P + (p < B % P)
        assert got["slice_bytes"] == [int(x) for x in st[p, 0]]
        assert got["slice_rbs"] == [int(x) for x in st[p, 1]]
        assert got["queued_bytes"] == [int(x) for x in bs[p, 0]]
        assert got["dropped_bytes"] == [int(x) for x in bs[p, 1]]
        assert got["records"] == [int(x) for x in bs[p, 2]]
    assert bs[:, 0].sum() > 0 and bs[:, 1].sum() > 0 and bs[:, 2].sum() > 0   # queues left, drops, records held
    assert bs[0, :, 0].sum() == 0                                                # slice 0 of config 0 is backlogged


CASES = [(9, False, 1, 1), (9, False, 2, 1), (9, True, 1, 1), (9, True, 2, 1), (9, False, 2, 2), (8, True, 2, 1),
         (10, False, 2, 1), (7, False, 2, 2), (11, False, 1, 1), (101, False, 1, 2), (103, True, 2, 1), (1, False, 1, 1)]


@pytest.mark.parametrize("algo,replay,nb,P", CASES)
def test_closed_loop_batch_equals_python_mirror(algo, replay, nb, P, tmp_path):
    B, T, seed, log_cell = 19, 45, 6, 7
    cfgs, trafs = zip(*[_files(tmp_path, nb, tag=str(p),
                               groups=GROUPS if p == 0 else [(n, w, (a, b, 1 - e, s)) for n, w, (a, b, e, s) in GROUPS[::-1]],
                               traffic=TRAFFIC if p == 0 else TRAFFIC[::-1]) for p in range(P)])
    args = ["--algo", algo, "--cells", B, "--ttis", T, "--seed", seed, "--buffers", K, "--log-cell", log_cell,
            "--log-prefix", tmp_path / "cell"]
    for c, t in zip(cfgs, trafs):
        args += ["--config", c, "--traffic", t]
    rep = None
    if replay:
        targs, traces, mp, n_rows = _traces(tmp_path)
        args += targs
        rep = (traces, mp, n_rows)
    lines = _run(*args)
    st, bs, out, err = mirror(algo, cfgs, trafs, B, T, seed, log_cell, rep)
    check_lines(lines, st, bs, B, P)
    assert (tmp_path / "cell.stdout").read_text() == out
    assert (tmp_path / "cell.stderr").read_text() == err
    assert err.count("\n") > T
    if algo in (8, 9, 101, 103) and nb == 1:
        assert "hol_delay: 0.0" in err   # finite queues with a delay show in the log


def test_one_traffic_file_for_every_config(tmp_path):
    """--traffic once with two --config: the file applies to both."""
    c0, t0 = _files(tmp_path, 1, tag="a")
    c1, _ = _files(tmp_path, 1, tag="b", groups=[(n, w * 0.5, q) for n, w, q in GROUPS])
    B, T = 12, 30
    lines = _run("--algo", 9, "--cells", B, "--ttis", T, "--seed", 3, "--buffers", K, "--config", c0, "--config", c1,
                 "--traffic", t0)
    st, bs, _, _ = mirror(9, [c0, c1], [t0, t0], B, T, 3, 0)
    check_lines(lines, st, bs, B, 2)


def test_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: rs_batch --gpus 2 --buffers is compared with --gpus 1 only where two are present")
    cfg, traffic = _files(tmp_path, 2)
    runs = []
    for n in (1, 2):
        runs.append(_run("--algo", 9, "--config", cfg, "--traffic", traffic, "--buffers", K, "--cells", 301, "--ttis", 64,
                         "--seed", 3, "--gpus", n, "--log-cell", 200, "--log-prefix", tmp_path / f"c{n}")[0])
    for k in ("slice_bytes", "slice_rbs", "queued_bytes", "dropped_bytes", "records"):
        assert runs[0][k] == runs[1][k], k
    assert runs[1]["gpus"] == 2 and sum(runs[0]["queued_bytes"]) > 0
    for ext in ("stdout", "stderr"):   # cell 200 lives on GPU 1
        assert (tmp_path / f"c1.{ext}").read_text() == (tmp_path / f"c2.{ext}").read_text()

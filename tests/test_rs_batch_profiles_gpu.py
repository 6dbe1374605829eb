"""GPU: rs_batch with a repeated --config (slice profiles): cell b uses config b % P, one output line per config, and
the totals equal Scheduler.from_profiles on the same seeded inputs.  With one --config the output is what it was."""
import json
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

pytestmark = pytest.mark.gpu
BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")


def _config(path, groups, ues):
    cfg = {"slices": [{"n_slices": n, "weight": w, "algo_alpha": a, "algo_beta": b, "algo_epsilon": e, "algo_psi": p}
                      for n, w, (a, b, e, p) in groups], "ues_per_slice": ues}
    path.write_text(json.dumps(cfg, indent=2))
    return str(path)


def _run(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    r = subprocess.run([BIN, *[str(a) for a in args]], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    return [json.loads(x) for x in r.stdout.strip().splitlines()]


def _configs(tmp_path):
    a = _config(tmp_path / "a.json", [(3, 0.2, (0, 0, 1, 1)), (2, 0.2, (0, 0, 1, 0))], [4, 2, 6, 1, 3])
    b = _config(tmp_path / "b.json", [(2, 0.35, (0, 0, 2, 1)), (3, 0.1, (0, 0, 0, 1))], [1, 7, 3, 3, 2])
    c = _config(tmp_path / "c.json", [(5, 0.2, (0, 0, 1, 1))], [3, 3, 3, 3, 4])
    return [a, b, c]


@pytest.mark.parametrize("algo", [9, 8, 7, 1, 10, 11, 101, 103])
def test_repeated_config_equals_from_profiles(algo, tmp_path):
    B, T, seed, log_cell = 37, 35, 4, 13   # cell 13 uses config 13 % 3 = 1
    paths = _configs(tmp_path)
    args = ["--algo", algo, "--cells", B, "--ttis", T, "--seed", seed, "--log-cell", log_cell,
            "--log-prefix", tmp_path / "cell"]
    got = _run(*[x for p in paths for x in ("--config", p)], *args)
    profiles = [sched.load_slice_config(p) for p in paths]
    P, S, U, G = len(paths), len(profiles[0][0]), len(profiles[0][2]), 64
    cp = np.arange(B) % P
    g = sched.Scheduler.from_profiles(algo, profiles, cp, cqi_per_rb=2)
    cqi = workload.synth_cqi(seed, 0, B, 0, T, U, G)
    draws = (workload.synth_rand_draws(seed, 0, B, 0, T, S, g.rand_stride) if algo == 11
             else workload.synth_rand2(seed, 0, B, 0, T, S))
    _, dts = workload.tti_clock(T)
    res = g.run_host(sched.pack_cqi(cqi), draws, dts, want_aux=True, ttis_per_launch=16)
    st = g.get_stats()
    assert len(got) == P
    for p in range(P):
        assert got[p]["config"] == p and got[p]["config_file"] == paths[p]
        assert got[p]["cells"] == int((cp == p).sum()) and got[p]["batch_cells"] == B
        assert got[p]["slice_bytes"] == [int(x) for x in st[p, 0]], p
        assert got[p]["slice_rbs"] == [int(x) for x in st[p, 1]], p
        assert int(st[p, 1].sum()) > 0
    # the logged cell's text names its own config's slices
    lw = sched.LogWriter(algo, profiles[1][2], S, cqi_per_rb=2)
    for t in range(T):
        if algo == 10:
            lw.tti_grants(100 + t, sched.pack_cqi(cqi[t, log_cell]), int(res["alloc_n"][t, log_cell]),
                          res["alloc_ue"][t, log_cell], res["alloc_rbg"][t, log_cell], res["tbs_bits"][t, log_cell],
                          res["final_cqi"][t, log_cell], res["slice_target"][t, log_cell], res["slice_quota"][t, log_cell])
            continue
        lw.tti(100 + t, sched.pack_cqi(cqi[t, log_cell]), res["rbg_to_ue"][t, log_cell], res["tbs_bits"][t, log_cell],
               res["final_cqi"][t, log_cell] if algo != 1 else None,
               res["slice_target"][t, log_cell] if algo in (8, 9, 101, 103) else None,
               res["slice_quota"][t, log_cell] if algo in (8, 9, 101, 103) else None)
    assert (tmp_path / "cell.stdout").read_text() == lw.stdout
    assert (tmp_path / "cell.stderr").read_text() == lw.stderr
    g.close()


def test_one_config_prints_what_it_printed(tmp_path):
    paths = _configs(tmp_path)
    got = _run("--algo", 9, "--config", paths[0], "--cells", 20, "--ttis", 10)
    assert len(got) == 1 and "config" not in got[0] and got[0]["cells"] == 20


def test_configs_of_different_shapes_are_refused(tmp_path):
    paths = _configs(tmp_path)
    other = _config(tmp_path / "d.json", [(4, 0.25, (0, 0, 1, 1))], [4, 4, 4, 4])
    r = subprocess.run([BIN, "--algo", "9", "--config", paths[0], "--config", other, "--cells", "8", "--ttis", "2"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "every config must have the same" in r.stderr, r.stderr


def test_two_gpus_pass_each_shard_its_assignment(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    paths = _configs(tmp_path)
    cfg = [x for p in paths for x in ("--config", p)]
    one = _run("--algo", 9, *cfg, "--cells", 41, "--ttis", 20, "--seed", 2)
    two = _run("--algo", 9, *cfg, "--cells", 41, "--ttis", 20, "--seed", 2, "--gpus", 2)
    for a, b in zip(one, two):
        assert a["slice_bytes"] == b["slice_bytes"] and a["slice_rbs"] == b["slice_rbs"]

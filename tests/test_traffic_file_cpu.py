"""CPU: the traffic file of rs_batch --buffers / --traffic and sched.load_traffic_config, which reads it the same way,
and the 16.16 rate rule both take from rs_arrival_spec.  Every error is found before a handle exists, so rs_batch
reports it without a GPU."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg_two_bearers.json")   # 4 slice groups of 1, 2, 2, 1 slices; 19 UEs
GOOD = {"bearers": 2, "slices": [{"backlogged": 1}, {"pkt_bytes": 1500, "pkts_per_tti": 0.6},
                                 {"pkt_bytes": 300, "pkts_per_tti": 2.5}, {"backlogged": 1}]}


def _write(tmp_path, obj, name="traffic.json"):
    path = tmp_path / name
    path.write_text(obj if isinstance(obj, str) else json.dumps(obj))
    return str(path)


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "3", *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_rate_rule():
    assert sched.arrival_spec(1500, 0.6) == (1500, 39322)          # 39321.6 rounds up
    assert sched.arrival_spec(1500, 0.15) == (1500, 9830)          # 9830.4 rounds down
    assert sched.arrival_spec(200, 2.5) == (200, 163840)
    assert sched.arrival_spec(40, 0.5 / 65536 * 3) == (40, 2)      # 1.5 units: halves away from zero
    assert sched.arrival_spec(40, 1 / 65536) == (40, 1)
    assert sched.arrival_spec(0, 0) == (0, 0)
    assert sched.arrival_spec(0x7fffffff, 0.9) == (0x7fffffff, 58982)
    for pkt, rate, what in [(1500.5, 1, "pkt_bytes"), (-1, 1, "pkt_bytes"), (2 ** 31, 0, "pkt_bytes"),
                            (1500, -0.1, "pkts_per_tti"), (1500, float("nan"), "pkts_per_tti"),
                            (1500, float("inf"), "pkts_per_tti"), (1500, 32768, "16.16"), (1500, 1e-7, "1/65536"),
                            (10 ** 9, 3, "overflow int32"), (0x7fffffff, 1, "overflow int32")]:
        with pytest.raises(ValueError, match=what):
            sched.arrival_spec(pkt, rate)


def test_load_traffic_config(tmp_path):
    nb, bl, pkt, q16 = sched.load_traffic_config(_write(tmp_path, GOOD), CFG)
    _, _, u2s = sched.load_slice_config(CFG)
    assert nb == 2 and bl.shape == (19, 2) and bl.dtype == bool
    slice_bl = np.array([1, 0, 0, 0, 0, 1], bool)                   # the groups expanded by n_slices
    assert np.array_equal(bl, np.repeat(slice_bl[u2s][:, None], 2, axis=1))
    assert pkt.tolist() == [0, 1500, 1500, 300, 300, 0] and q16.tolist() == [0, 39322, 39322, 163840, 163840, 0]
    one = dict(GOOD, bearers=1)
    nb, bl, _, _ = sched.load_traffic_config(_write(tmp_path, one), CFG)
    assert nb == 1 and bl.shape == (19, 1)


BAD = [
    ({"slices": GOOD["slices"]}, '"bearers" must be 1 or 2'),
    (dict(GOOD, bearers=3), '"bearers" must be 1 or 2'),
    (dict(GOOD, slices={"backlogged": 1}), '"slices" must be a list'),
    (dict(GOOD, slices=GOOD["slices"][:3]), '3 entries in "slices", the slice config has 4 slice groups'),
    (dict(GOOD, slices=GOOD["slices"] + [{"backlogged": 1}]), '5 entries in "slices", the slice config has 4'),
    (dict(GOOD, slices=[{"backlogged": 0}] + GOOD["slices"][1:]), r'slices\[0\]: "backlogged" must be 1'),
    (dict(GOOD, slices=GOOD["slices"][:1] + [{"pkt_bytes": 1500}] + GOOD["slices"][2:]), r"slices\[1\]: expected"),
    (dict(GOOD, slices=GOOD["slices"][:1] + [{"pkt_bytes": 1500, "pkts_per_tti": 1, "backlogged": 1}] + GOOD["slices"][2:]),
     r"slices\[1\]: expected"),
    (dict(GOOD, slices=GOOD["slices"][:2] + [{"pkt_bytes": 1500.5, "pkts_per_tti": 1}] + GOOD["slices"][3:]),
     r"slices\[2\]: pkt_bytes 1500.5 is not an integer"),
    (dict(GOOD, slices=GOOD["slices"][:2] + [{"pkt_bytes": 1500, "pkts_per_tti": -2}] + GOOD["slices"][3:]),
     r"slices\[2\]: pkts_per_tti -2 is not a finite rate"),
    (dict(GOOD, slices=GOOD["slices"][:2] + [{"pkt_bytes": 1500, "pkts_per_tti": 40000}] + GOOD["slices"][3:]),
     r"slices\[2\]: pkts_per_tti 40000 does not fit 16.16"),
    (dict(GOOD, slices=GOOD["slices"][:2] + [{"pkt_bytes": 100000000, "pkts_per_tti": 30}] + GOOD["slices"][3:]),
     r"slices\[2\]: .*overflow int32"),
]


@pytest.mark.parametrize("obj,msg", BAD)
def test_bad_traffic_files(tmp_path, obj, msg):
    path = _write(tmp_path, obj)
    with pytest.raises(ValueError, match=msg):
        sched.load_traffic_config(path, CFG)
    r = _batch("--config", CFG, "--buffers", 8, "--traffic", path)
    assert r.returncode == 1 and r.stdout == ""
    assert r.stderr.startswith(f"rs_batch: traffic file {path}: ")
    assert re.search(msg, r.stderr), r.stderr


def test_argument_errors(tmp_path):
    path = _write(tmp_path, GOOD)
    cases = [(["--config", CFG, "--buffers", 8], "--buffers needs --traffic FILE"),
             (["--config", CFG, "--traffic", path], "--traffic needs --buffers K"),
             (["--config", CFG, "--buffers", 0, "--traffic", path], "--buffers K: K records per bearer, 1..65536"),
             (["--config", CFG, "--buffers", 65537, "--traffic", path], "1..65536"),
             (["--config", CFG, "--config", CFG, "--config", CFG, "--buffers", 8, "--traffic", path, "--traffic", path],
              "2 --traffic files for 3 --config files"),
             (["--config", CFG, "--buffers", 8, "--traffic", str(tmp_path / "none.json")], "Fail to open traffic file")]
    for args, msg in cases:
        r = _batch(*args)
        assert r.returncode == 1 and msg in r.stderr and r.stdout == "", (args, r.stderr)
    # traffic files of one batch must agree on the bearers per UE (one rs_config.n_bearers for every profile)
    one = _write(tmp_path, dict(GOOD, bearers=1), "one.json")
    r = _batch("--config", CFG, "--config", CFG, "--buffers", 8, "--traffic", path, "--traffic", one)
    assert r.returncode == 1 and 'traffic files with "bearers" 2 and 1' in r.stderr
    # the usage text names the new flags
    r = subprocess.run([BIN, "--algo", "9"], capture_output=True, text=True)
    assert r.returncode == 2 and "[--buffers K --traffic FILE ...]" in r.stderr


def test_valid_files_get_as_far_as_the_device(tmp_path):
    """Everything parses; without a GPU the run stops at the handle, with a GPU it runs (checked on the GPU)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_rs_batch_buffers_gpu.py runs it")
    r = _batch("--config", CFG, "--buffers", 8, "--traffic", _write(tmp_path, GOOD))
    assert r.returncode == 1 and "rs_create" in r.stderr and r.stdout == ""


def test_shipped_example_files():
    """tests/data/traffic20x5_ab.json with cfg20x5_ab.json (INTEGRATION.md section 4): the even slices alpha/beta and
    fed 1500-byte packets, the odd ones backlogged."""
    d = os.path.join(ROOT, "tests", "data")
    nb, bl, pkt, q16 = sched.load_traffic_config(os.path.join(d, "traffic20x5_ab.json"), os.path.join(d, "cfg20x5_ab.json"))
    _, p, u2s = sched.load_slice_config(os.path.join(d, "cfg20x5_ab.json"))
    s = np.arange(20)
    assert nb == 1 and np.array_equal(bl[:, 0], (u2s % 2 == 1))
    assert np.array_equal(pkt, np.where(s % 2 == 0, 1500, 0)) and np.array_equal(p[:, 0] == 1, s % 2 == 0)
    assert np.array_equal(q16, np.where(s % 2 == 1, 0, np.where(s % 4 == 0, 39322, 9830)))

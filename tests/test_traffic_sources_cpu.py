"""CPU: traffic sources (rs_set_sources / rs_synth_traffic, include/rs_sched.h) through their integer twin
workload.synth_traffic, the on-off rate rule rs_onoff_spec, and the periodic and on-off entries of the traffic file as
sched.load_traffic and rs_batch read them.  The twin is checked against a scalar, bearer-by-bearer statement of the
header's rules written here; the device is checked against the twin on the GPU (test_traffic_sources_gpu.py)."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import SRC_NONE, SRC_ONOFF, SRC_PERIODIC, SRC_RATE
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg_two_bearers.json")   # 4 slice groups of 1, 2, 2, 1 slices; 19 UEs
M64 = (1 << 64) - 1


# ---- the header's rules, one bearer at a time, in Python integers ----------------------------------------------------
def _sm(x):
    z = (x + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def bearer_ref(seed, cell, ue, slot, src, tti0, n, on=None):
    """(arrivals [n], ON state after the last TTI) of one bearer running source `src` from TTI tti0."""
    key_arr = _sm((seed & 0xFFFFFFFF) | (0x41525200 << 32))   # "ARR\0": rs_synth_arrivals' key
    key_src = _sm((seed & 0xFFFFFFFF) | (0x53524300 << 32))   # "SRC\0"
    ctr = ((cell << 20) ^ (ue << 8) ^ slot ^ (((ue >> 12) * 0xD6E8FEB86659FD93) & M64)) & M64
    hb = _sm(ctr ^ key_src)
    lo, kind = hb & 0xFFFFFFFF, src["kind"]
    period = src.get("period_ttis", 1)
    phi = (hb >> 32) % period
    if kind == SRC_ONOFF and on is None:
        on = lo < (src["leave_off_q32"] << 32) // (src["leave_on_q32"] + src["leave_off_q32"])
    out = []
    for tau in range(tti0, tti0 + n):
        draw = _sm((((tau << 40) & M64) ^ ctr) ^ key_arr)
        if kind == SRC_RATE:
            q = src["pkts_q16"]
            out.append(src["pkt_bytes"] * ((q >> 16) + ((draw >> 48) < (q & 0xFFFF))))
        elif kind == SRC_PERIODIC:
            fr = src["frame_bytes"]
            out.append(fr[((tau + phi) // period + lo % len(fr)) % len(fr)] if (tau + phi) % period == 0 else 0)
        elif kind == SRC_ONOFF:
            if (draw & 0xFFFFFFFF) < (src["leave_on_q32"] if on else src["leave_off_q32"]):
                on = not on
            out.append(src["pkt_bytes"] if on and (tau + phi) % period == 0 else 0)
        else:
            out.append(0)
    return out, on


def _phase(seed, cell, ue, slot, period):
    key_src = _sm((seed & 0xFFFFFFFF) | (0x53524300 << 32))
    return (_sm(((cell << 20) ^ (ue << 8) ^ slot) ^ key_src) >> 32) % period


ON, OFF = sched.onoff_spec(4, 6)
SOURCES = [{"kind": SRC_NONE},
           {"kind": SRC_RATE, "pkt_bytes": 300, "pkts_q16": sched.arrival_spec(300, 1.3)[1]},
           {"kind": SRC_PERIODIC, "period_ttis": 7, "frame_bytes": [5000, 600, 700]},
           {"kind": SRC_ONOFF, "pkt_bytes": 90, "period_ttis": 3, "leave_on_q32": ON, "leave_off_q32": OFF}]
U2S = np.array([0, 1, 2, 3, 2, 3], dtype=np.int32)


def test_onoff_rule():
    assert sched.onoff_spec(2, 2 ** 32) == (2 ** 31, 1)
    assert sched.onoff_spec(1000, 1500) == (4294967, 2863312)          # 4294967.296 down, 2863311.53 up
    m = 2 ** 32 / 2.5
    assert 2 ** 32 / m == 2.5 and sched.onoff_spec(m, m) == (3, 3)       # halves away from zero
    for on, off, what in [(1.999, 10, "on_ttis 1.999"), (10, 0, "off_ttis 0"), (-5, 10, "on_ttis -5"),
                          (float("nan"), 10, "on_ttis nan"), (10, float("inf"), "off_ttis inf"),
                          (2 ** 32 + 1, 10, "on_ttis 4.29497e\\+09")]:
        with pytest.raises(ValueError, match=what + r" is not a finite mean in \[2, 2\^32\] TTIs"):
            sched.onoff_spec(on, off)


@pytest.mark.parametrize("nb", [1, 2])
def test_twin_equals_the_rules_bearer_by_bearer(nb):
    seed, cell0, B, tti0, T = 11, 5, 3, 40, 70
    arr, st = workload.synth_traffic(seed, cell0, B, tti0, T, U2S, SOURCES, n_bearers=nb)
    assert arr.shape == ((T, B, 6) if nb == 1 else (T, B, 6, 2)) and arr.dtype == np.int32
    a = arr.reshape(T, B, 6, nb)
    s = st.reshape(B, 6, nb)
    for b in range(B):
        for u in range(6):
            for i in range(nb):
                want, on = bearer_ref(seed, cell0 + b, u, i, SOURCES[U2S[u]], tti0, T)
                assert a[:, b, u, i].tolist() == want, (b, u, i)
                assert s[b, u, i] == (bool(on) if U2S[u] == 3 else 0)
    for k in (1, 2, 3):
        assert (a[:, :, U2S == k] > 0).any()                       # every kind draws something here


def test_rate_is_synth_arrivals():
    q = np.array([[0, 9830, 39322, 3 * 65536 + 7]], dtype=np.int32)
    pkt = np.array([[0, 1500, 200, 40]], dtype=np.int32)
    src = [{"kind": SRC_RATE, "pkt_bytes": int(p), "pkts_q16": int(x)} for p, x in zip(pkt[0], q[0])]
    for nb in (1, 2):
        got, _ = workload.synth_traffic(3, 7, 5, 11, 30, U2S % 4, src, n_bearers=nb)
        assert np.array_equal(got, workload.synth_arrivals(3, 7, 5, 11, 30, U2S % 4, pkt, q, n_bearers=nb))


def test_periodic_frames():
    frames = [9000, 100, 200, 300, 400]
    src = [{"kind": SRC_PERIODIC, "period_ttis": 10, "frame_bytes": frames}]
    B, U, T, seed = 40, 5, 200, 4
    arr, _ = workload.synth_traffic(seed, 0, B, 0, T, np.zeros(U, np.int32), [src[0]], n_bearers=2)
    phases = set()
    for b in range(B):
        for u in range(U):
            for i in range(2):
                x = arr[:, b, u, i]
                hit = np.flatnonzero(x)
                assert len(hit) == T // 10 and np.all(np.diff(hit) == 10)          # one frame per period
                phi = _phase(seed, b, u, i, 10)
                assert (hit[0] + phi) % 10 == 0
                phases.add(hit[0])
                k = frames.index(x[hit[0]])                                        # per-bearer start ...
                assert x[hit].tolist() == [frames[(k + j) % 5] for j in range(len(hit))]   # ... then in order
    assert len(phases) == 10                                                       # phases spread over the period


def test_onoff_arrivals_fall_on_aligned_on_ttis():
    src = [{"kind": SRC_ONOFF, "pkt_bytes": 33, "period_ttis": 4, "leave_on_q32": ON, "leave_off_q32": OFF}]
    B, U, T, seed = 20, 5, 300, 8
    arr, _ = workload.synth_traffic(seed, 2, B, 5, T, np.zeros(U, np.int32), src)
    assert set(np.unique(arr)) == {0, 33}
    for b in range(B):
        for u in range(U):
            phi = _phase(seed, 2 + b, u, 0, 4)
            tau = 5 + np.flatnonzero(arr[:, b, u])
            assert np.all((tau + phi) % 4 == 0)
    # and on ON TTIs only: with a period of one TTI the arrivals are the ON indicator itself
    one = [dict(src[0], period_ttis=1)]
    a1, _ = workload.synth_traffic(seed, 2, B, 5, T, np.zeros(U, np.int32), one)
    assert np.all(a1[arr > 0] > 0) and (a1 > arr).any()


def test_chunked_calls_equal_one_call():
    whole, st = workload.synth_traffic(21, 3, 4, 7, 200, U2S, SOURCES, n_bearers=2)
    parts, s = [], None
    for k in range(10):
        a, s = workload.synth_traffic(21, 3, 4, 7 + 20 * k, 20, U2S, SOURCES, n_bearers=2, state=s)
        parts.append(a)
    assert np.array_equal(np.concatenate(parts), whole) and np.array_equal(s, st)


def test_cell_shards_equal_the_whole():
    whole, st = workload.synth_traffic(5, 0, 8, 0, 50, U2S, SOURCES)
    a, sa = workload.synth_traffic(5, 0, 3, 0, 50, U2S, SOURCES)
    b, sb = workload.synth_traffic(5, 3, 5, 0, 50, U2S, SOURCES)
    assert np.array_equal(np.concatenate([a, b], axis=1), whole) and np.array_equal(np.concatenate([sa, sb]), st)


def test_two_bearers_draw_independently():
    src = [{"kind": SRC_ONOFF, "pkt_bytes": 1, "period_ttis": 1, "leave_on_q32": ON, "leave_off_q32": OFF}]
    arr, _ = workload.synth_traffic(9, 0, 50, 0, 400, np.zeros(4, np.int32), src, n_bearers=2)
    one, _ = workload.synth_traffic(9, 0, 50, 0, 400, np.zeros(4, np.int32), src)
    assert np.array_equal(arr[..., 0], one)                       # slot 0 is the one-bearer draw
    x, y = arr[..., 0].reshape(-1).astype(float), arr[..., 1].reshape(-1).astype(float)
    assert abs(np.corrcoef(x, y)[0, 1]) < 0.02 and (x != y).mean() > 0.3


def test_profiles_pick_their_rows():
    rows = [SOURCES, SOURCES[::-1], [SOURCES[2]] * 4]
    u2s = np.stack([U2S, U2S[::-1], U2S])
    cp = np.array([2, 0, 1, 1, 0, 2, 2])
    arr, st = workload.synth_traffic(6, 10, 7, 3, 40, u2s, rows, n_bearers=2, cell_profile=cp)
    for b, p in enumerate(cp):
        a1, s1 = workload.synth_traffic(6, 10 + b, 1, 3, 40, u2s[p], rows[p], n_bearers=2)
        assert np.array_equal(arr[:, b], a1[:, 0]) and np.array_equal(st[b], s1[0])


def test_onoff_long_run_statistics():
    """ON fraction and mean ON / OFF run lengths of 20000 TTIs x 150 bearers, against the spec (50 / 150 TTIs).  A long
    window keeps the run cut off at its end (counted as a whole run here) under 1 % of the runs."""
    on_q, off_q = sched.onoff_spec(50, 150)
    src = [{"kind": SRC_ONOFF, "pkt_bytes": 1, "period_ttis": 1, "leave_on_q32": on_q, "leave_off_q32": off_q}]
    for seed in (1, 2):
        arr, _ = workload.synth_traffic(seed, 0, 30, 0, 20000, np.zeros(5, np.int32), src)
        x = arr.reshape(20000, -1).T.astype(np.int8)
        assert abs(x.mean() / 0.25 - 1) < 0.03
        # mean run length = TTIs spent in a state / runs of that state (a run starts at TTI 0 or at a change)
        starts = np.concatenate([np.ones((x.shape[0], 1), bool), np.diff(x, axis=1) != 0], axis=1)
        mean_on = (x == 1).sum() / (starts & (x == 1)).sum()
        mean_off = (x == 0).sum() / (starts & (x == 0)).sum()
        assert abs(mean_on / 50 - 1) < 0.03, mean_on
        assert abs(mean_off / 150 - 1) < 0.03, mean_off


# ---- traffic files ---------------------------------------------------------------------------------------------------
VIDEO = {"period_ttis": 40, "frame_bytes": [30000, 5000, 5000, 9000]}
VOICE = {"pkt_bytes": 40, "period_ttis": 20, "on_ttis": 1000, "off_ttis": 1500}
MIXED = {"bearers": 2, "slices": [{"backlogged": 1}, VIDEO, VOICE, {"pkt_bytes": 300, "pkts_per_tti": 2.5}]}


def _write(tmp_path, obj, name="traffic.json"):
    path = tmp_path / name
    path.write_text(obj if isinstance(obj, str) else json.dumps(obj))
    return str(path)


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "3", *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_load_traffic(tmp_path):
    nb, bl, src = sched.load_traffic(_write(tmp_path, MIXED), CFG)
    _, _, u2s = sched.load_slice_config(CFG)
    assert nb == 2 and bl.shape == (19, 2)
    assert np.array_equal(bl, np.repeat(np.array([1, 0, 0, 0, 0, 0], bool)[u2s][:, None], 2, axis=1))
    on, off = sched.onoff_spec(1000, 1500)
    assert src == [{"kind": SRC_NONE}] + [{"kind": SRC_PERIODIC, "period_ttis": 40, "frame_bytes": VIDEO["frame_bytes"]}] * 2 + \
        [{"kind": SRC_ONOFF, "pkt_bytes": 40, "period_ttis": 20, "leave_on_q32": on, "leave_off_q32": off}] * 2 + \
        [{"kind": SRC_RATE, "pkt_bytes": 300, "pkts_q16": 163840}]
    # the rate-only reader keeps its results for rate files and points to load_traffic for the new forms
    with pytest.raises(ValueError, match="load_traffic"):
        sched.load_traffic_config(_write(tmp_path, MIXED), CFG)
    rate = dict(MIXED, slices=[{"backlogged": 1}, {"pkt_bytes": 1500, "pkts_per_tti": 0.6}] * 2)
    nb, bl2, pkt, q16 = sched.load_traffic_config(_write(tmp_path, rate), CFG)
    _, bl3, src3 = sched.load_traffic(_write(tmp_path, rate), CFG)
    assert np.array_equal(bl2, bl3) and pkt.tolist() == [s.get("pkt_bytes", 0) for s in src3]
    assert q16.tolist() == [0, 39322, 39322, 0, 0, 39322]


def _with(entry, g=1):
    s = list(MIXED["slices"])
    s[g] = entry
    return dict(MIXED, slices=s)


BAD = [
    (_with({"period_ttis": 40}), r"slices\[1\]: expected"),
    (_with({"period_ttis": 40, "frame_bytes": 5000}), r"slices\[1\]: expected"),
    (_with({"frame_bytes": [5000]}), r"slices\[1\]: expected"),
    (_with({"period_ttis": 0, "frame_bytes": [100]}), r"slices\[1\]: period_ttis 0 is not an integer 1\.\.2147483647"),
    (_with({"period_ttis": 2.5, "frame_bytes": [100]}), r"slices\[1\]: period_ttis 2.5 is not an integer"),
    (_with({"period_ttis": 40, "frame_bytes": []}), r"slices\[1\]: 0 frame_bytes, expected 1\.\.1024"),
    (_with({"period_ttis": 40, "frame_bytes": [1] * 1025}), r"slices\[1\]: 1025 frame_bytes, expected 1\.\.1024"),
    (_with({"period_ttis": 40, "frame_bytes": [100, 0]}), r"slices\[1\]: frame_bytes 0 is not an integer 1\.\."),
    (_with({"period_ttis": 40, "frame_bytes": [2 ** 31]}), r"slices\[1\]: frame_bytes 2.14748e\+09 is not an integer"),
    (_with({"pkt_bytes": 40, "period_ttis": 20, "on_ttis": 1000}, 2), r"slices\[2\]: expected"),
    (_with(dict(VOICE, frame_bytes=[1]), 2), r"slices\[2\]: expected"),
    (_with({"pkt_bytes": 40, "pkts_per_tti": 1, "period_ttis": 20}, 2), r"slices\[2\]: expected"),
    (_with(dict(VOICE, pkt_bytes=0), 2), r"slices\[2\]: pkt_bytes 0 is not an integer 1\.\."),
    (_with(dict(VOICE, period_ttis=-3), 2), r"slices\[2\]: period_ttis -3 is not an integer 1\.\."),
    (_with(dict(VOICE, on_ttis=1), 2), r"slices\[2\]: on_ttis 1 is not a finite mean in \[2, 2\^32\] TTIs"),
    (_with(dict(VOICE, off_ttis=1e10), 2), r"slices\[2\]: off_ttis 1e\+10 is not a finite mean"),
]


@pytest.mark.parametrize("obj,msg", BAD)
def test_bad_entries_refused_by_both_readers(tmp_path, obj, msg):
    path = _write(tmp_path, obj)
    with pytest.raises(ValueError, match=msg):
        sched.load_traffic(path, CFG)
    r = _batch("--config", CFG, "--buffers", 8, "--traffic", path)
    assert r.returncode == 1 and r.stdout == ""
    assert r.stderr.startswith(f"rs_batch: traffic file {path}: ")     # refused before a handle exists
    assert re.search(msg, r.stderr), r.stderr


def test_new_forms_get_as_far_as_the_device(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_traffic_sources_gpu.py runs rs_batch on these forms")
    r = _batch("--config", CFG, "--buffers", 8, "--traffic", _write(tmp_path, MIXED))
    assert r.returncode == 1 and "rs_create" in r.stderr and r.stdout == ""


def test_shipped_video_voice_example():
    """tests/data/traffic20x5_video_voip.json with cfg20x5_ab.json (INTEGRATION.md section 4): periodic frames and on-off
    sources on the alpha/beta slices, the others backlogged."""
    d = os.path.join(ROOT, "tests", "data")
    nb, bl, src = sched.load_traffic(os.path.join(d, "traffic20x5_video_voip.json"), os.path.join(d, "cfg20x5_ab.json"))
    _, p, u2s = sched.load_slice_config(os.path.join(d, "cfg20x5_ab.json"))
    kinds = np.array([s["kind"] for s in src])
    assert nb == 1 and np.array_equal(bl[:, 0], u2s % 2 == 1)
    s = np.arange(20)
    assert np.array_equal(kinds, np.where(s % 2 == 1, SRC_NONE, np.where(s % 4 == 0, SRC_PERIODIC, SRC_ONOFF)))
    assert np.all(p[kinds != SRC_NONE, :2] == 1)                          # every source feeds an alpha/beta slice
    arr, _ = workload.synth_traffic(1, 0, 8, 0, 400, u2s, src)
    assert (arr[:, :, u2s % 4 == 0] > 0).any() and (arr[:, :, u2s % 4 == 2] > 0).any() and not arr[:, :, u2s % 2 == 1].any()

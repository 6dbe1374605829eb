"""GPU: the drop-in itself.  The product's host plug-in (radiosaber_b200/host/rs_gpu_scheduler.h -> C ABI -> CUDA)
installed in place of the reference scheduler class (ids 1, 7, 8, 9, 10, 11, 101, 103) must reproduce, record for record,
what the reference classes produced on the same CQI / rand() inputs (tests/golden).

Where oracle/_ref/ref_harness_gpu is built (it needs the reference LTE-Sim sources, which are not part of this repository)
the plug-in runs inside the reference's own SingleCellWithI scenario.  Otherwise build/dropin/dropin_replay runs the same
header against the stand-in LTE-Sim classes of oracle/dropin/ltesim.h, fed each TTI with what the record says the
simulator handed the reference scheduler (clock, CQI, queues, head-of-line delays, rand() values); the bearers' rates and
counters and the slice state chain on their own from the first TTI, and the record is compared field for field.  The
two-bearer cell is replayed from per-bearer records and compared through its log text.  Which path ran is named in
every failure message."""
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import workload
from tests.helpers import ROOT, load_golden
from tools import golden_io

pytestmark = pytest.mark.gpu
HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness_gpu")   # make -C oracle ref gpu REF=<reference source tree>
REPLAY = os.path.join(ROOT, "build", "dropin", "dropin_replay")       # make -C oracle dropin (__graft_entry__.build())


def write_replay(path, now, cqi, exists, app_id, avg0, tx0, last0, state0, queue, hol, draws):
    """dropin_replay's --replay file (layout in oracle/dropin/dropin_replay.cpp); per-bearer arrays are [..][U][NB]."""
    T, U, G = cqi.shape
    NB = exists.shape[1]
    with open(path, "wb") as f:
        # PacketScheduler counts TTIs from the start of the run: 1 ms each
        f.write(np.array([T, U, len(state0), G, NB, int(round(now[0] * 1000))], "<i4").tobytes())
        f.write(exists.astype(np.uint8).tobytes() + app_id.astype("<i4").tobytes())
        f.write(avg0.astype("<f8").tobytes() + tx0.astype("<i4").tobytes())
        f.write(np.float64(last0).tobytes() + np.asarray(state0, "<f8").tobytes())
        f.write(np.ascontiguousarray(cqi, dtype=np.uint8).tobytes())
        for t in range(T):
            f.write(np.float64(now[t]).tobytes())
            f.write((queue[t] > 0).astype(np.uint8).tobytes() + queue[t].astype("<i4").tobytes() + hol[t].astype("<f8").tobytes())
            f.write(np.array([len(draws[t])], "<i4").tobytes() + np.asarray(draws[t], "<i4").tobytes())


def scripted_draws(rec, algo):
    """The rand() values the reference's DoSchedule drew, per TTI (ids 1 and 7 draw none)."""
    if algo == 11:
        return [rec["rand_ng"][t, :int(rec["rand_ng_n"][t])] for t in range(int(rec["T"]))]
    if algo in (8, 9, 10, 101, 103):
        return list(rec["rand2"])
    return [np.zeros(0)] * int(rec["T"])


def write_replay_inputs(path, rec):
    """dropin_replay's --replay file from a golden record: one bearer per UE."""
    T, U = int(rec["T"]), int(rec["U"])
    queue = rec["queue"] if "queue" in rec else np.full((T, U), 100000000, np.int32)
    hol = rec["hol"] if "hol" in rec else np.zeros((T, U))
    write_replay(path, rec["now"], rec["cqi"], np.ones((U, 1)), np.arange(U)[:, None], rec["avg_before"][0][:, None],
                 rec["tx_before"][0][:, None], rec["now"][0] - rec["dt"][0], rec["state_before"][0], queue[:, :, None],
                 hol[:, :, None], scripted_draws(rec, int(rec["algo"])))


CASES = ["a9_fix20x5_synth", "a9_diffw_synth", "a9_diffw_trace", "a9_small_synth", "a8_fix20x5_synth", "a8_small_synth",
         "a7_fix20x5_synth", "a7_mix20_synth", "a7_small_synth", "a1_fix20x5_synth", "a1_small_synth",
         # finite queues and head-of-line delays (internet flows): the plug-in reads them from the bearers
         "a9_qif_synth", "a8_qif_synth", "a7_qif_synth", "a1_qif_synth",
         # the other inter-slice algorithms of DownlinkTransportScheduler: UpperBound (grants as a list), SubOpt, Vogel
         "a10_fix20x5_synth", "a10_diffw_synth", "a10_small_synth", "a10_qif_synth",
         "a101_fix20x5_synth", "a101_diffw_synth", "a101_small_synth", "a101_qif_synth",
         "a103_fix20x5_synth", "a103_diffw_synth", "a103_small_synth", "a103_qif_synth",
         # NVS non-greedy: the plug-in takes 300 x (listed users of the served slice) rand() values per TTI from the process
         "a11_fix20x5_synth", "a11_small_synth", "a11_qif_synth"]


@pytest.mark.parametrize("name", CASES)
def test_plugin_inside_lte_sim_matches_reference(name, tmp_path):
    rec = load_golden(name)
    S, U, T = int(rec["S"]), int(rec["U"]), int(rec["T"])
    cfg = {"slices": [], "ues_per_slice": [int((rec["ue_to_slice"] == s).sum()) for s in range(S)]}
    for s in range(S):
        a, b, e, p = (int(x) for x in rec["params"][s])
        cfg["slices"].append({"n_slices": 1, "weight": float(rec["weight"][s]), "video_app": 0, "video_bitrate": 0,
                              "internet_flow": 0, "if_bitrate": 0, "backlog_flow": 1, "algo_alpha": a,
                              "algo_beta": b, "algo_epsilon": e, "algo_psi": p})
    if "queue" in rec:   # the traffic mix is part of the scenario: the recorded run's own config
        cfg = json.loads(str(rec["config_json"]))
    (tmp_path / "cfg.json").write_text(json.dumps(cfg))
    assert int(rec["cqi_per_rb"]) == 0
    np.ascontiguousarray(rec["cqi"], dtype=np.uint8).tofile(tmp_path / "cqi.bin")
    np.ascontiguousarray(rec["rand2"], dtype=np.int32).tofile(tmp_path / "rand.bin")
    out = tmp_path / "rec.bin"
    algo = int(rec["algo"])
    extra = ["--alloc-log", str(tmp_path / "alloc.bin")] if algo == 10 else []
    if algo == 11:
        extra = ["--rand-log", str(tmp_path / "draws.bin")]
    # which path ran is part of every failure message: inside the reference's LTE-Sim, or the stand-in replay (where the
    # rand() values are the record's own, so rand2 checks only that the plug-in draws them in the same number and order)
    how = "reference LTE-Sim" if os.path.exists(HARNESS) else "stand-in replay"
    name = f"{name} ({how})"
    if os.path.exists(HARNESS):
        cmd = [HARNESS, "--gpu", "--ttis", str(T), "--cqi", str(tmp_path / "cqi.bin"), "--rand", str(tmp_path / "rand.bin"),
               "--seed", str(int(rec["seed"]))]
    else:
        assert os.path.exists(REPLAY), "build/dropin/dropin_replay missing: run __graft_entry__.build()"
        write_replay_inputs(tmp_path / "replay.bin", rec)
        cmd = [REPLAY, "--replay", str(tmp_path / "replay.bin")]
    r = subprocess.run(cmd + ["--algo", str(algo), "--config", str(tmp_path / "cfg.json"), "--out", str(out)] + extra,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (name, r.stdout[-500:], r.stderr[-500:])
    got = golden_io.compact(golden_io.parse_record_stream(str(out)))
    assert int(got["T"]) == T, name
    fields = ["rbg_to_ue", "bits", "final_cqi", "avg_before", "avg_after", "tx_after", "cum_bytes", "cum_rbs",
              "state_before", "state_after", "dt"]
    if algo in (8, 9, 10, 101, 103):
        fields += ["target", "quota", "rand2"]
    if algo in (7, 11):
        fields += ["nvs_slice"]
    for f in fields:
        assert np.array_equal(np.asarray(got[f]), np.asarray(rec[f])), (name, f)
    if algo == 11:   # every rand() value drawn inside DoSchedule: the same count and the same values as the reference's
        raw = np.fromfile(tmp_path / "draws.bin", dtype="<i4")
        pos = 0
        for t in range(T):
            k = int(raw[pos])
            assert k == int(rec["rand_ng_n"][t]), (name, t)
            assert np.array_equal(raw[pos + 1:pos + 1 + k], rec["rand_ng"][t, :k]), (name, t)
            pos += 1 + k
        assert pos == len(raw)
    if algo == 10:   # every (user, RBG) grant of every TTI, in the order of the users' RB lists
        raw = np.fromfile(tmp_path / "alloc.bin", dtype="<i2")
        pos = 0
        for t in range(T):
            k = int(raw[pos]) | (int(raw[pos + 1]) << 16)
            pairs = raw[pos + 2:pos + 2 + 2 * k].reshape(k, 2)
            pos += 2 + 2 * k
            assert k == int(rec["alloc_n"][t]), (name, t)
            assert np.array_equal(pairs[:, 0], rec["alloc_ue"][t, :k]) and np.array_equal(pairs[:, 1], rec["alloc_rbg"][t, :k]), (name, t)
        assert pos == len(raw)


# ---- two bearers per UE (internet_flow: 2) ---------------------------------------------------------------------
# The record format is per UE, so here the golden is the reference's own log text: the plug-in must print the same
# allocation dump (stdout) and the same per-bearer cumu_bytes / cumu_rbs lines (stderr) -- which only happens if every
# TTI's allocation, every bearer's share of the bytes and, through the bearers' own EWMA, every later TTI are identical.
# Inside the reference's LTE-Sim: tests/golden/logs_two_bearers (tools/make_golden_logs_two_bearers.py).  Stand-in replay:
# the per-bearer records of tests/golden/two_bearers (tools/make_golden_two_bearers.py; every bearer's queue and
# head-of-line delay per TTI, application ids) with the reference's text of the same run beside them, plus every
# bearer's rate and byte / RB counters after each TTI.
TWO_BEARER_LOGS = os.path.join(ROOT, "tests", "golden", "logs_two_bearers")
TWO_BEARER_RECS = os.path.join(ROOT, "tests", "golden", "two_bearers")


def _scheduler_lines(text):
    """Drop what is not scheduler output: the RLC's "ipflow end ..." lines and the inter-slice function's all_bytes."""
    return [l for l in text.splitlines() if not l.startswith("ipflow ") and not l.startswith("all_bytes")]


def _compare_logs(want_text, got_text, T, what):
    want, got = _scheduler_lines(want_text), _scheduler_lines(got_text)
    assert len(want) > T, what
    for k, (a, b) in enumerate(zip(want, got)):
        assert a == b, (what, k, a, b)
    assert len(got) == len(want), what


@pytest.mark.parametrize("algo", [9, 8, 7, 10, 101, 103])
def test_two_bearers_per_ue_inside_lte_sim(algo, tmp_path):
    from tools import make_golden_logs_two_bearers as mb
    cfg = json.load(open(mb.CFG))
    if os.path.exists(HARNESS):
        cqi, rnd = mb.write_inputs(str(tmp_path), cfg)
        cmd = mb.command(HARNESS, algo, cqi, rnd, str(tmp_path / "got"), cfg)
        r = subprocess.run(cmd[:1] + ["--gpu"] + cmd[1:], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (r.stdout[-500:], r.stderr[-500:])
        for ext in ("stdout", "stderr"):
            _compare_logs(open(os.path.join(TWO_BEARER_LOGS, f"a{algo}.{ext}")).read(), (tmp_path / f"got.{ext}").read_text(),
                          mb.TTIS, (algo, ext, "reference LTE-Sim"))
        return

    assert os.path.exists(REPLAY), "build/dropin/dropin_replay missing: run __graft_entry__.build()"
    rec = golden_io.load_npz(os.path.join(TWO_BEARER_RECS, f"a{algo}.npz"))
    T, U, G = int(rec["T"]), int(rec["U"]), int(rec["G"])
    now, dts = workload.tti_clock(T)    # the reference's clock from 0.1 s, when the applications start
    assert np.array_equal(dts, rec["dt"])
    cqi = workload.synth_cqi(int(rec["seed"]), 0, 1, 0, T, U, G)[:, 0]
    write_replay(tmp_path / "replay.bin", now, cqi, rec["exists"], rec["app_id"], rec["avg_before"][0], rec["tx_before"][0],
                 now[0] - dts[0], rec["state_before"][0], rec["queue"], rec["hol"], scripted_draws(rec, algo))
    extra = ["--alloc-log", str(tmp_path / "alloc.bin")] if algo == 10 else []
    r = subprocess.run([REPLAY, "--replay", str(tmp_path / "replay.bin"), "--algo", str(algo), "--config", mb.CFG,
                        "--out", str(tmp_path / "rec.bin"), "--bearer-out", str(tmp_path / "bearers.bin"),
                        "--log-out", str(tmp_path / "got")] + extra, capture_output=True, text=True, timeout=600)
    what = (algo, "stand-in replay")
    assert r.returncode == 0, (what, r.stdout[-500:], r.stderr[-500:])
    for ext in ("stdout", "stderr"):
        with gzip.open(os.path.join(TWO_BEARER_RECS, f"a{algo}.{ext}.gz"), "rt") as f:
            _compare_logs(f.read(), (tmp_path / f"got.{ext}").read_text(), T, what + (ext,))
    got = golden_io.parse_record_stream(str(tmp_path / "rec.bin"))
    fields = ["bits", "final_cqi", "state_after"] + (["rbg_to_ue"] if algo != 10 else [])
    fields += ["target", "quota"] if algo != 7 else ["nvs_slice"]
    for f in fields:
        assert np.array_equal(np.asarray(got[f]), np.asarray(rec[f])), what + (f,)
    post = np.dtype([("avg", "<f8"), ("tx", "<i4"), ("pad", "<i4"), ("cum_bytes", "<u8"), ("cum_rbs", "<u8")])
    per_bearer = np.fromfile(tmp_path / "bearers.bin", dtype=post).reshape(T, U, 2)
    ex = rec["exists"].astype(bool)
    for k, gk in (("avg", "avg_after"), ("tx", "tx_after"), ("cum_bytes", "cum_bytes"), ("cum_rbs", "cum_rbs")):
        assert np.array_equal(per_bearer[k][:, ex], rec[gk][:, ex]), what + (gk,)

"""CPU: the synthetic channel (rs_set_channels / rs_synth_channel, include/rs_sched.h) through its integer twin
workload.synth_channel, the float -> integer rule of rs_channel_spec, and the channel file of rs_batch --channel, which
sched.load_channel reads the same way.  Every file error is found before a handle exists, so rs_batch reports it without
a GPU."""
import json
import math
import os
import re
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from radiosaber_b200.workload import CH_FADING, CH_IID, splitmix64
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg_two_bearers.json")   # 4 slice groups of 1, 2, 2, 1 slices; 19 UEs
COUNTS = [0, 0, 1, 2, 5, 9, 14, 20, 25, 20, 14, 9, 5, 2, 0]
FADE = sched.channel_spec(COUNTS, 1.5, 6, 4)
IID = {"kind": CH_IID}


def _ref_cqi(seed, cell, ue, e, g, ch):
    """One sample by the rules of include/rs_sched.h, in Python integers."""
    m = (1 << 64) - 1
    sm = lambda x: int(splitmix64(np.array([x & m], dtype=np.uint64))[0])   # noqa: E731
    fold = ((ue >> 12) * 0xD6E8FEB86659FD93) & m
    if ch["kind"] == CH_IID:
        key = int(workload._key(seed, workload.DOMAIN_CQI))
        u32 = sm((((e & m) << 40) ^ (cell << 20) ^ (ue << 8) ^ g ^ fold) & m ^ key) >> 32
        return 1 + sum(u32 >= t for t in workload.CQI_CDF32.tolist())
    key = int(workload._key(seed, workload.DOMAIN_CHANNEL))
    d = [sm(((cell << 20) ^ (ue << 8) ^ i ^ fold) ^ key) for i in range(17)]
    hi, lo = [x >> 32 for x in d], [x & 0xFFFFFFFF for x in d]

    def slope(raw, coh):
        w = (1 << 31) // coh if coh else 0
        return (((raw * (2 * w + 1)) >> 32) - w) % (1 << 32)

    level = 1 + sum(hi[0] >= t for t in ch["level_thr"])
    tab = workload.cos_q14().tolist()
    x = 0
    for k in range(8):
        ph = (hi[1 + k] + g * slope(lo[1 + k], ch["coherence_rbgs"]) + (e % (1 << 32)) * slope(hi[9 + k], ch["coherence_epochs"]))
        x += tab[(ph % (1 << 32)) >> 22]
    return min(max(level + ((x * ch["depth_q8"] + (1 << 22)) >> 23), 1), 15)


def test_cos_table_equals_the_committed_include():
    text = open(os.path.join(ROOT, "include", "rs_cos_q14.inc")).read()
    body = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    vals = [int(v) for v in body.replace(",", " ").split()]
    assert vals == workload.cos_q14().tolist()
    assert len(vals) == 1024 and vals[0] == 16384 and vals[512] == -16384 and vals[256] == 0


@pytest.mark.parametrize("U", [7, 4100])
def test_twin_equals_the_rules_sample_by_sample(U):
    """Per-profile rows, IID and FADING slices, cells from 5000, epochs past 2^32 (uint32 wrap), UEs past 4096 (fold)."""
    u2s = np.stack([np.arange(U) % 3, (np.arange(U) + 1) % 3]).astype(np.int32)
    flat = sched.channel_spec(COUNTS, 2.0, 0, 0)
    rows = [[FADE, IID, flat], [IID, dict(FADE, coherence_rbgs=1, coherence_epochs=3), FADE]]
    cp = np.array([1, 0, 1])
    e0 = (1 << 32) - 2
    got = workload.synth_channel(9, 5000, 3, e0, 4, u2s, rows, cell_profile=cp, n_rbgs=48)
    assert got.shape == (4, 3, U, 48) and got.dtype == np.uint8
    rng = np.random.default_rng(U)
    ues = sorted(set(rng.integers(0, U, 12).tolist()) | ({U - 1, 4096, 4097} & set(range(U))))
    for j in range(4):
        for b in range(3):
            for u in ues:
                ch = rows[cp[b]][u2s[cp[b], u]]
                for g in (0, 1, 17, 47):
                    assert got[j, b, u, g] == _ref_cqi(9, 5000 + b, u, e0 + j, g, ch), (j, b, u, g)
    if U > 4096:   # UE u and u + 4096 share the low 12 bits of the counter: the fold keeps them apart
        assert not np.array_equal(got[:, :, 3], got[:, :, 4099])


def test_all_iid_is_synth_cqi():
    u2s = np.arange(11) % 4
    want = workload.synth_cqi(4, 20, 6, 7, 5, 11, 64)
    assert np.array_equal(workload.synth_channel(4, 20, 6, 7, 5, u2s, [IID] * 4), want)
    mixed = workload.synth_channel(4, 20, 6, 7, 5, u2s, [IID, FADE, IID, FADE])
    iid = u2s % 2 == 0
    assert np.array_equal(mixed[:, :, iid], want[:, :, iid]) and not np.array_equal(mixed[:, :, ~iid], want[:, :, ~iid])


def test_depth_zero_is_the_level_and_levels_follow_the_counts():
    counts = np.array([0, 3, 0, 10, 20, 40, 60, 80, 60, 40, 20, 10, 5, 2, 1], dtype=np.float64)
    ch = sched.channel_spec(counts, 0, 5, 5)
    assert ch["depth_q8"] == 0
    B, U = 1000, 100
    got = workload.synth_channel(3, 0, B, 11, 3, np.zeros(U, np.int32), [ch], n_rbgs=16)
    assert (got == got[:1, :, :, :1]).all()                     # every RBG and epoch is the UE's level
    obs = np.bincount(got[0, :, :, 0].reshape(-1), minlength=16)[1:].astype(np.float64)
    exp = counts / counts.sum() * B * U
    assert obs[exp == 0].sum() == 0                              # levels without counts never occur
    k = exp > 0
    chi2 = float(((obs[k] - exp[k]) ** 2 / exp[k]).sum())
    assert chi2 < 36.1                                           # 12 degrees of freedom: p = 0.0003


def _corr(a, b):
    a = a - a.mean()
    b = b - b.mean()
    return float((a * b).mean() / np.sqrt((a * a).mean() * (b * b).mean()))


@pytest.mark.parametrize("coh_f,coh_t", [(8, 6), (4, 10)])
def test_offset_spread_and_correlation_are_the_stated_sinc_product(coh_f, coh_t):
    """x before depth, rounding and clamping: standard deviation 2^15 within 2 %, autocorrelation at lags 1, coh / 2 and
    coh in RBGs and in epochs within 0.03 of sinc(pi lag / coh)."""
    n_e = coh_t + 1
    x = workload.channel_offset_sum(12, 0, 400, 3, n_e, 100, 64, coh_f, coh_t).astype(np.float64)
    assert abs(x.std() / 2 ** 15 - 1) < 0.02
    for lag in (1, coh_f // 2, coh_f):
        assert abs(_corr(x[..., :-lag], x[..., lag:]) - math.sin(math.pi * lag / coh_f) / (math.pi * lag / coh_f)) < 0.03
    for lag in (1, coh_t // 2, coh_t):
        assert abs(_corr(x[:-lag], x[lag:]) - math.sin(math.pi * lag / coh_t) / (math.pi * lag / coh_t)) < 0.03
    # both lags at once: the product
    want = np.sinc(2 / coh_f) * np.sinc(1 / coh_t)
    assert abs(_corr(x[:-1, ..., :-2], x[1:, ..., 2:]) - want) < 0.03


def test_coherence_zero_is_flat_or_frozen():
    flat = workload.channel_offset_sum(5, 0, 30, 0, 6, 20, 64, 0, 3)
    assert (flat == flat[..., :1]).all() and not (flat == flat[:1]).all()
    frozen = workload.channel_offset_sum(5, 0, 30, 0, 6, 20, 64, 3, 0)
    assert (frozen == frozen[:1]).all() and not (frozen == frozen[..., :1]).all()
    both = workload.synth_channel(5, 0, 30, 100, 4, np.zeros(20), [sched.channel_spec(COUNTS, 3, 0, 0)])
    assert (both == both[:1, :, :, :1]).all()


def test_shards_and_chunks_equal_one_call():
    u2s = np.arange(9) % 3
    rows = [FADE, IID, dict(FADE, coherence_epochs=0)]
    whole = workload.synth_channel(2, 100, 12, 40, 10, u2s, rows)
    parts = [workload.synth_channel(2, 100 + c0, n, 40 + e0, m, u2s, rows)
             for c0, n in ((0, 5), (5, 7)) for e0, m in ((0, 3), (3, 7))]
    assert np.array_equal(np.concatenate([np.concatenate(parts[:2], 0), np.concatenate(parts[2:], 0)], 1), whole)


def test_profiles_pick_their_rows():
    u2s = np.stack([np.arange(8) % 2, 1 - np.arange(8) % 2])
    cp = np.array([0, 1, 1, 0, 1])
    flat = sched.channel_spec(COUNTS, 1, 0, 0)
    got = workload.synth_channel(6, 0, 5, 0, 2, u2s, [[FADE, IID], [FADE, flat]], cell_profile=cp)
    want = [workload.synth_channel(6, 0, 5, 0, 2, u2s[0], [FADE, IID]),
            workload.synth_channel(6, 0, 5, 0, 2, u2s[1], [FADE, flat])]
    assert not np.array_equal(want[0], want[1])
    for b in range(5):
        assert np.array_equal(got[:, b], want[cp[b]][:, b])


def test_channel_spec_rule():
    ch = sched.channel_spec([1] * 15, 1.5, 8, 3)
    assert ch["kind"] == CH_FADING and ch["depth_q8"] == 384
    assert ch["level_thr"] == [((k + 1) << 32) // 15 for k in range(14)]
    assert (ch["coherence_rbgs"], ch["coherence_epochs"]) == (8, 3)
    c = [0] * 15
    c[4] = 7
    assert sched.channel_spec(c, 0, 0, 0)["level_thr"] == [0] * 4 + [0xFFFFFFFF] * 10   # level 5 only (2^-32 above)
    assert sched.channel_spec(c, 1.5 / 256, 1.5, 2.5)["depth_q8"] == 2                  # halves away from zero
    assert sched.channel_spec(c, 1.5 / 256, 1.5, 2.5)["coherence_rbgs"] == 2
    assert sched.channel_spec(c, 1.5 / 256, 1.5, 2.5)["coherence_epochs"] == 3
    assert sched.channel_spec(c, 15, 2 ** 31 - 1, 1)["depth_q8"] == 3840
    big = [0] * 14 + [2 ** 32 - 1]
    assert sched.channel_spec(big, 1, 1, 1)["level_thr"] == [0] * 14
    for counts, d, f, t, what in [([1.5] + [1] * 14, 1, 1, 1, r"level_counts\[0\] = 1.5 is not an integer"),
                                  ([1] * 14 + [-1], 1, 1, 1, r"level_counts\[14\] = -1"),
                                  ([float("nan")] * 15, 1, 1, 1, r"level_counts\[0\] = nan"),
                                  ([0] * 15, 1, 1, 1, "sum to 0"), ([2 ** 31] * 2 + [0] * 13, 1, 1, 1, "sum to 4294967296"),
                                  ([1] * 15, -0.5, 1, 1, "depth_cqi -0.5"), ([1] * 15, 15.01, 1, 1, "depth_cqi 15.01"),
                                  ([1] * 15, float("inf"), 1, 1, "depth_cqi inf"),
                                  ([1] * 15, 1, 0.5, 1, "coherence_rbgs 0.5 is not 0 or in"),
                                  ([1] * 15, 1, -1, 1, "coherence_rbgs -1"), ([1] * 15, 1, 1, 2 ** 31, "coherence_epochs 2.14"),
                                  ([1] * 15, 1, 1, float("nan"), "coherence_epochs nan")]:
        with pytest.raises(ValueError, match=what):
            sched.channel_spec(counts, d, f, t)


# ---- the channel file ------------------------------------------------------------------------------------------------
SPEC = {"level_counts": COUNTS, "depth_cqi": 1.5, "coherence_rbgs": 6, "coherence_reports": 4}
GOOD = {"note": "read by neither reader", "report_ttis": 40, "slices": [{"iid": 1}, SPEC, dict(SPEC, depth_cqi=0), {"iid": 1}]}


def _write(tmp_path, obj, name="channel.json"):
    path = tmp_path / name
    path.write_text(obj if isinstance(obj, str) else json.dumps(obj))
    return str(path)


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "3", *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_load_channel(tmp_path):
    rep, ch = sched.load_channel(_write(tmp_path, GOOD), CFG)
    fade = sched.channel_spec(COUNTS, 1.5, 6, 4)
    assert rep == 40 and ch == [IID, fade, fade, dict(fade, depth_q8=0), dict(fade, depth_q8=0), IID]
    rep, ch = sched.load_channel(_write(tmp_path, {"slices": [{"iid": 1}] * 4}), CFG)
    assert rep == 1 and ch == [IID] * 6
    rep, ch = sched.load_channel(_write(tmp_path, {"report_ttis": None, "slices": [{"iid": 1}] * 4}), CFG)
    assert rep == 1 and ch == [IID] * 6


def _with(entry, g=1, **top):
    doc = dict(GOOD, **top)
    doc["slices"] = list(GOOD["slices"])
    if entry is not None:
        doc["slices"][g] = entry
    return doc


BAD = [
    ("[1, 2]", '"slices" must be a list'),
    ({"report_ttis": 40, "slices": {"iid": 1}}, '"slices" must be a list'),
    (_with(None, report_ttis=0), r'"report_ttis" must be an integer 1\.\.2147483647'),
    (_with(None, report_ttis=2.5), r'"report_ttis" must be an integer'),
    (_with(None, report_ttis=2 ** 31), r'"report_ttis" must be an integer'),
    (dict(GOOD, slices=GOOD["slices"][:3]), r'3 entries in "slices", the slice config has 4 slice groups'),
    (_with({"iid": 2}), r'slices\[1\]: "iid" must be 1'),
    (_with({"iid": 2}, report_ttis=None), r'slices\[1\]: "iid" must be 1'),        # a null report_ttis is 1 for both
    (_with({"iid": 1, "depth_cqi": 1}), r"slices\[1\]: expected"),
    (_with(dict(SPEC, level_counts=COUNTS[:14])), r"slices\[1\]: expected"),
    (_with({k: v for k, v in SPEC.items() if k != "coherence_reports"}), r"slices\[1\]: expected"),
    (_with(dict(SPEC, coherence_epochs=4)), r"slices\[1\]: expected"),
    (_with(dict(SPEC, level_counts=[1.5] + COUNTS[1:]), 2), r"slices\[2\]: level_counts\[0\] = 1.5 is not an integer"),
    (_with(dict(SPEC, level_counts=[0] * 15), 2), r"slices\[2\]: level_counts sum to 0"),
    (_with(dict(SPEC, depth_cqi=16), 2), r"slices\[2\]: depth_cqi 16 is not in \[0, 15\]"),
    (_with(dict(SPEC, coherence_rbgs=0.25), 2), r"slices\[2\]: coherence_rbgs 0.25 is not 0 or in \[1, 2147483647\]"),
    (_with(dict(SPEC, coherence_reports=-2), 2), r"slices\[2\]: coherence_epochs -2 is not 0 or in"),
]


@pytest.mark.parametrize("obj,msg", BAD)
def test_bad_files_refused_by_both_readers(tmp_path, obj, msg):
    path = _write(tmp_path, obj)
    with pytest.raises(ValueError, match=msg):
        sched.load_channel(path, CFG)
    r = _batch("--config", CFG, "--channel", path)
    assert r.returncode == 1 and r.stdout == ""
    assert r.stderr.startswith(f"rs_batch: channel file {path}: ")      # refused before a handle exists
    assert re.search(msg, r.stderr), r.stderr


def test_argument_errors(tmp_path):
    path = _write(tmp_path, GOOD)
    other = _write(tmp_path, dict(GOOD, report_ttis=7), "other.json")
    for args, msg in [(["--config", CFG, "--channel", path, "--traces", tmp_path, "--mapping", path],
                       "--channel and --traces both give the CQI"),
                      (["--config", CFG, "--config", CFG, "--config", CFG, "--channel", path, "--channel", path],
                       "2 --channel files for 3 --config files"),
                      (["--config", CFG, "--config", CFG, "--channel", path, "--channel", other],
                       'channel files with "report_ttis" 40 and 7'),
                      (["--config", CFG, "--channel", tmp_path / "missing.json"], "Fail to open channel file")]:
        r = _batch(*args)
        assert r.returncode == 1 and msg in r.stderr, r.stderr


def test_valid_files_get_as_far_as_the_device(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_channel_gpu.py runs rs_batch on these files")
    r = _batch("--config", CFG, "--channel", _write(tmp_path, GOOD))
    assert r.returncode == 1 and "rs_create" in r.stderr and r.stdout == ""


def test_shipped_example_file():
    """tests/data/channel20x5_traces.json (INTEGRATION.md section 4) is what tools/fit_channel_traces.py fits to the
    committed trace subset, and reads as one FADING channel for every slice of cfg20x5.json, reported every 40 TTIs."""
    from tools import fit_channel_traces
    d = os.path.join(ROOT, "tests", "data")
    path = os.path.join(d, "channel20x5_traces.json")
    with open(path) as f:
        doc = json.load(f)
    entry, _ = fit_channel_traces.fit(np.load(os.path.join(ROOT, "tests", "golden", "traces", "trace_subset.npz"))["rows"])
    assert doc["slices"] == [entry] and "not a validated channel model" in doc["note"]
    assert sum(entry["level_counts"]) == 127
    rep, ch = sched.load_channel(path, os.path.join(d, "cfg20x5.json"))
    assert rep == 40 and len(ch) == 20 and all(c["kind"] == CH_FADING for c in ch)
    cqi = workload.synth_channel(1, 0, 64, 0, 4, np.repeat(np.arange(20), 5), ch)
    means = cqi.reshape(4, 64 * 100, 64).mean(axis=(0, 2))
    assert 4 < np.percentile(means, 10) < np.percentile(means, 90) < 14          # cell-edge and cell-centre UEs

"""Trace-driven CQI ingest (SURVEY section 8 row a16; enb-mac-entity.cc:42-56, 160-193).

CPU: the oracle's ingest restatement and the library's host-side parsers against the CQI the
unmodified reference ingested (golden *_trace records) and against each other.
GPU: the trace-driven kernels through the C ABI against the reference records and the oracle."""
import os

import numpy as np
import pytest

from oracle import trace_ingest as ti
from oracle.pyoracle import OracleScheduler
from radiosaber_b200 import sched, workload
from tests.helpers import GOLDEN, load_golden

FIX = os.path.join(GOLDEN, "traces", "trace_subset.npz")
# the reference's own trace files (a RadioSaber checkout named by RS_REFERENCE), for the provenance check of the fixture
REF_TRACES = os.path.join(os.environ["RS_REFERENCE"], "cqi-traces-noise0") if os.environ.get("RS_REFERENCE") else ""
TRACE_GOLDENS = ["a9_fix20x5_trace", "a8_fix20x5_trace", "a7_fix20x5_trace", "a1_fix20x5_trace", "a9_diffw_trace",
                 "a10_fix20x5_trace", "a11_fix20x5_trace"]


def _fixture():
    z = np.load(FIX)
    ids = z["trace_ids"]
    slot = {int(t): k for k, t in enumerate(ids)}
    return z["mapping"], ids, z["rows"], slot


def _ue_trace_slots(mapping, slot, U, rec=None):
    """Fixture slot of the trace each UE replays.  A UE whose CQI reports never reached the eNB in the
    recorded run (its record shows the initial all-10 vector on every TTI, ENodeB.cpp:207-217; UE 0 of
    the id 7/8 records) is marked -1."""
    out = np.array([slot[ti.trace_of_ue(mapping, u)] for u in range(U)], dtype=np.int32)
    if rec is not None:
        out[(rec["cqi"] == ti.INITIAL_CQI).all(axis=(0, 2))] = -1
    return out


@pytest.mark.parametrize("name", TRACE_GOLDENS)
def test_oracle_ingest_reproduces_reference_cqi(name):
    """mapping[u % n], line (int)(Now*1000/40) % 475 of the last report, reports every 40 TTIs from the
    first scheduled TTI: exactly the CQI vectors the reference's scheduler saw."""
    rec = load_golden(name)
    mapping, ids, rows, slot = _fixture()
    U, T = int(rec["U"]), int(rec["T"])
    ue_slot = _ue_trace_slots(mapping, slot, U, rec)
    assert (ue_slot < 0).sum() <= 1
    tr = ti.rows_for_run(rec["now"], 0)
    assert tr.max() < rows.shape[1]
    for t in range(T):
        assert np.array_equal(ti.cqi_at(rows, ue_slot[None], int(tr[t]))[0], rec["cqi"][t]), t


def test_host_row_formula_matches_oracle():
    now, _ = workload.tti_clock(3000)
    for t in now[::7]:
        assert sched.trace_row(t) == ti.trace_row(t)
    for x in (0.0, 0.039999999, 0.04, 18.999999, 19.0, 19.04, 1234.5678):
        assert sched.trace_row(x) == ti.trace_row(x)
    rec = load_golden("a9_fix20x5_trace")
    assert np.array_equal(sched.trace_rows_for_run(rec["now"], 0), ti.rows_for_run(rec["now"], 0))
    assert np.array_equal(sched.trace_rows_for_run(rec["now"], 13), ti.rows_for_run(rec["now"], 13))


def test_parsers_round_trip(tmp_path):
    """Files written in the reference's text format parse identically through the library's C parser and
    the oracle's restatement (short lines repeat the last value, like operator>> leaves it)."""
    mapping, ids, rows, slot = _fixture()
    rng = np.random.default_rng(5)
    per_rb = np.repeat(rows[3], 8, axis=1)            # [8][512]
    per_rb[5, 100:108] = rng.integers(1, 16, 8)      # a line that varies inside an RBG
    p = tmp_path / "ue7.log"
    lines = [" ".join(str(int(v)) for v in r) for r in per_rb]
    lines[6] = " ".join(lines[6].split()[:500])        # short line
    p.write_text("\n".join(lines) + "\n")
    a = sched.parse_trace_file(str(p), n_rows=8, n_rbs=512)
    b = ti.read_trace(str(p), n_rows=8, n_rbs=512)
    assert np.array_equal(a, b)
    assert np.array_equal(a[:6], per_rb[:6])
    assert (a[6, 500:] == a[6, 499]).all()
    m = tmp_path / "mapping.config"
    m.write_text("".join(f"{i} {int(t)}\n" for i, t in enumerate(mapping)))
    assert np.array_equal(sched.parse_mapping_file(str(m)), mapping)
    assert np.array_equal(ti.read_mapping(str(m)), mapping)
    tr, got = sched.load_trace_dir(str(tmp_path), n_rows=8)
    assert got.tolist() == [7] and np.array_equal(tr[0], a)


@pytest.mark.skipif(not os.path.isdir(REF_TRACES), reason="needs the reference's cqi-traces-noise0 files (RS_REFERENCE=<checkout>), "
                    "which are not part of this repository: the fixture's provenance and the full-file parse go unchecked")
def test_fixture_equals_reference_files():
    mapping, ids, rows, slot = _fixture()
    assert np.array_equal(sched.parse_mapping_file(os.path.join(REF_TRACES, "mapping1.config")), mapping)
    for k in (0, len(ids) // 2, len(ids) - 1):
        full = sched.parse_trace_file(os.path.join(REF_TRACES, f"ue{int(ids[k])}.log"))
        assert full.shape == (475, 512)
        assert np.array_equal(full[:rows.shape[1], ::8], rows[k])
        assert np.array_equal(full, ti.read_trace(os.path.join(REF_TRACES, f"ue{int(ids[k])}.log")))


# ---- GPU ---------------------------------------------------------------------------------------------
FIELDS = ("rbg_to_ue", "tbs_bits", "mcs", "final_cqi")


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRACE_GOLDENS)
@pytest.mark.parametrize("layout", [0, 2])
def test_cuda_trace_run_matches_reference_record(name, layout):
    """One cell replaying cqi-traces-noise0 through mapping1.config on the device == what the unmodified
    reference produced from its own ingest of the same files."""
    rec = load_golden(name)
    mapping, ids, rows, slot = _fixture()
    algo, U, T = int(rec["algo"]), int(rec["U"]), int(rec["T"])
    g = sched.Scheduler(algo, rec["weight"], rec["params"], rec["ue_to_slice"], 1, cqi_per_rb=layout)
    g.set_traces(np.repeat(rows, 8, axis=2), _ue_trace_slots(mapping, slot, U, rec)[None])
    g.set_state(avg_rate=rec["avg_before"][0][None], tx_bytes=rec["tx_before"][0][None],
                slice_offset=rec["state_before"][0][None] if algo in (8, 9, 10) else None,
                nvs_ewma=rec["state_before"][0][None] if algo in (7, 11) else None)
    tr = sched.trace_rows_for_run(rec["now"], 0)
    draws = rec["rand_ng"] if algo == 11 else rec["rand2"]
    out = g.run_traces_host(tr, draws[:, None, :], rec["dt"], want_aux=True, ttis_per_launch=7)
    assert np.array_equal(out["rbg_to_ue"][:, 0], rec["rbg_to_ue"])
    assert np.array_equal(out["tbs_bits"][:, 0], rec["bits"])
    if algo != 1:
        assert np.array_equal(out["final_cqi"][:, 0], rec["final_cqi"])
    st = g.get_state()
    assert np.array_equal(st["avg_rate"][0], rec["avg_after"][-1])
    assert np.array_equal(st["cum_bytes"][0], rec["cum_bytes"][-1])
    assert np.array_equal(st["cum_rbs"][0], rec["cum_rbs"][-1])
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [9, 8, 7, 1])
@pytest.mark.parametrize("layout", [0, 1, 2])
def test_cuda_trace_batch_matches_oracle(algo, layout):
    """A batch whose cells each draw their own UE->trace mapping (Monte Carlo trace mappings), reports
    starting at TTI 3 (CQI 10 before), some bearers idle: device trace replay == oracle fed with the
    expanded CQI."""
    S, n, B, T = 6, 4, 37, 50
    rng = np.random.default_rng(100 + algo + layout)
    u2s = np.repeat(np.arange(S), n).astype(np.int32)
    U, G = S * n, 64
    w = rng.dirichlet(np.ones(S))
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    p[::2, 3] = 0
    n_tr, n_rows = 9, 11
    if layout == 1:   # per-RB traces that vary inside an RBG
        traces = rng.integers(1, 16, (n_tr, n_rows, 512)).astype(np.uint8)
    else:
        traces = np.repeat(rng.integers(1, 16, (n_tr, n_rows, G)).astype(np.uint8), 8, axis=2)
    ue_trace = rng.integers(-1, n_tr, (B, U)).astype(np.int32)
    now, dts = workload.tti_clock(T)
    # reports from TTI 3 on, every 5 TTIs; the line each report selects is drawn at random here (a 50 ms
    # run would only ever see lines 2 and 3 of a real trace)
    tr = np.repeat(rng.integers(0, n_rows, T // 5 + 1), 5)[:T].astype(np.int32)
    tr[:3] = -1
    active = (rng.random((T, B, U)) < 0.9).astype(np.uint8)
    active[:, 5] = 0
    rand2 = workload.synth_rand2(3, 0, B, 0, T, S)
    g = sched.Scheduler(algo, w, p, u2s, B, cqi_per_rb=layout)
    g.set_traces(traces, ue_trace)
    o = OracleScheduler(algo, w, p, u2s, B, cqi_per_rb=1 if layout == 1 else 0)
    out = g.run_traces_host(tr, rand2, dts, active=active, want_aux=True, ttis_per_launch=8)
    otab = traces if layout == 1 else traces[:, :, ::8]
    for t in range(T):
        ref = o.step(ti.cqi_at(otab, ue_trace, int(tr[t])), rand2[t], dt=float(dts[t]), active=active[t], want_aux=True)
        for k in FIELDS:
            assert np.array_equal(out[k][t], ref[k]), (t, k)
    sa, sb = g.get_state(), o.get_state()
    for k in ("avg_rate", "tx_bytes", "cum_bytes", "cum_rbs"):
        assert np.array_equal(sa[k], sb[k]), k
    g.close()


@pytest.mark.gpu
def test_cuda_trace_errors():
    S = 2
    u2s = np.array([0, 0, 1], dtype=np.int32)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    g = sched.Scheduler(9, [0.5, 0.5], p, u2s, 2, cqi_per_rb=0)
    _, dts = workload.tti_clock(2)
    with pytest.raises(sched.RsError):   # no traces loaded
        g.run_traces_host(np.zeros(2, np.int32), np.zeros((2, 2, 2), np.int32), dts)
    bad = np.full((1, 3, 512), 7, dtype=np.uint8)
    bad[0, 1, 9] = 8
    with pytest.raises(sched.RsError):   # varies inside an RBG under a per-RBG layout
        g.set_traces(bad, np.zeros((2, 3), np.int32))
    g.set_traces(np.full((1, 3, 512), 7, dtype=np.uint8), np.zeros((2, 3), np.int32))
    with pytest.raises(sched.RsError):   # row outside the table
        g.run_traces_host(np.array([0, 3], np.int32), np.zeros((2, 2, 2), np.int32), dts)
    g.close()

#!/usr/bin/env python3
"""Randomised differential run: CUDA path against the CPU oracle on random slice configurations, shapes,
CQI layouts, idle bearers, finite queues and head-of-line delays, several hundred TTIs each so that the
state (EWMA rates, offsets, credits) drifts far from its initial values.  Development / soak tool; the unit
tests under tests/ are the contract.  Usage: python tools/fuzz_parity.py [--seconds 120] [--seed 1] [--wide] [--limits]

--wide also draws the RBG count from the LTE-Sim bands, two bearers per UE, cells of up to ~600 UEs (512-thread
CTAs) and the multi-TTI entries (rs_run_host / rs_run_traces_host with a random launch length) instead of rs_step.

--limits draws near the limits rs_create accepts instead: every id, 24..64 slices, the bands, up to a few thousand UEs
and id 10's whole grant list (up to S*G grants, rs_set_grant_list_len)."""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import trace_ingest as ti  # noqa: E402
from oracle.pyoracle import OracleScheduler  # noqa: E402
from radiosaber_b200 import sched, workload  # noqa: E402


# (n_rbs, rbg_size) of the LTE-Sim bands as the plug-in trims them, 100 MHz and 64 RBGs of one RB
BANDS = [(6, 1), (14, 2), (24, 2), (48, 3), (72, 4), (100, 4), (256, 8), (504, 8), (64, 1), (512, 8)]


def _limits_draws(rng):
    """The configuration of a --limits case: (algo, S, u2s, w, p, layout, B, T, R, rbg)."""
    algo = int(rng.choice([1, 7, 8, 9, 10, 11, 101, 103]))
    S = int(rng.integers(24, 65))
    ues = rng.integers(1, 13, S)
    if rng.random() < 0.5:   # 480 .. 3000 UEs: 512 threads, per-thread UE loops
        ues = np.maximum(1, np.round(ues * rng.integers(480, 3000) / ues.sum())).astype(np.int64)
    u2s = np.repeat(np.arange(S), ues).astype(np.int32)
    w = rng.dirichlet(np.ones(S) * rng.choice([0.3, 0.5, 1.0]))
    p = np.zeros((S, 4), dtype=np.int32)
    p[:, 0] = rng.integers(0, 2, S)
    p[:, 1] = rng.integers(0, 2, S)
    p[:, 2] = rng.choice([0, 1, 1, 1, 2], S)
    p[:, 3] = rng.integers(0, 2, S)
    R, rbg = BANDS[int(rng.integers(0, len(BANDS)))]
    layout = int(rng.choice([0, 1, 2]))
    if layout == 2 and (R // rbg) % 8:
        layout = 0
    return algo, S, u2s, w, p, layout, int(rng.integers(1, 5)), int(rng.integers(60, 121)), R, rbg


def one_case(rng, case, wide=False, limits=False):
    """One random configuration; None or a description of the first mismatch.  wide=False draws exactly what it
    always has (the seeds of tests/test_fuzz_gpu.py keep their cases); wide=True adds the draws of --wide after them;
    limits=True then replaces the configuration with one of --limits (the earlier draws are still made)."""
    algo = int(rng.choice([9, 9, 9, 8, 7, 1, 10, 11, 101, 103]))
    S = int(rng.integers(1, 33))
    ues = rng.integers(1, 9 if algo == 11 else 13, S)
    if rng.random() < 0.15:
        ues[int(rng.integers(0, S))] = int(rng.integers(20, 60))
    u2s = np.repeat(np.arange(S), ues).astype(np.int32)
    U, G = len(u2s), 64
    w = rng.dirichlet(np.ones(S) * rng.choice([0.3, 1.0, 5.0]))
    p = np.zeros((S, 4), dtype=np.int32)
    p[:, 0] = rng.integers(0, 2, S)
    p[:, 1] = rng.integers(0, 2, S)
    p[:, 2] = rng.choice([0, 1, 1, 1, 2], S)
    p[:, 3] = rng.integers(0, 2, S)
    layout = int(rng.choice([0, 0, 1, 2]))
    B = int(rng.integers(1, 24))
    T = int(rng.integers(40, 260))
    queue_aware = rng.random() < 0.4
    with_active = rng.random() < 0.3
    R, rbg, nb, entry, tpl = 512, 8, 1, "step", 1
    if wide:
        R, rbg = BANDS[int(rng.integers(0, len(BANDS)))]
        G = R // rbg
        if layout == 2 and G % 8:
            layout = 0
        if algo != 1 and rng.random() < 0.3:
            nb, queue_aware = 2, True
        if algo != 11 and rng.random() < 0.3:   # a cell of 480..600 UEs: 512 threads (id 11: 300 draws per user)
            ues = np.maximum(1, np.round(ues * rng.integers(480, 600) / ues.sum())).astype(np.int64)
            while ues.sum() < 480:
                ues[int(rng.integers(0, S))] += 1
            u2s = np.repeat(np.arange(S), ues).astype(np.int32)
            U = len(u2s)
            B, T = min(B, 4), min(T, 60)
        entry = str(rng.choice(["step", "host", "trace"]))
        tpl = int(rng.integers(1, 65))
    grants = None
    if limits:
        algo, S, u2s, w, p, layout, B, T, R, rbg = _limits_draws(rng)
        U, G, nb = len(u2s), R // rbg, 1
        queue_aware = rng.random() < 0.5
        with_active = rng.random() < 0.3
        entry = str(rng.choice(["step", "host", "trace"]))
        tpl = int(rng.integers(1, 65))
        grants = max(S * G, 2 * G) if algo == 10 else None
    g = sched.Scheduler(algo, w, p, u2s, B, n_rbs=R, rbg_size=rbg, cqi_per_rb=layout, n_bearers=nb)
    if grants:
        g.set_grant_list_len(grants)
    o = OracleScheduler(algo, w, p, u2s, B, n_rbs=R, rbg_size=rbg, cqi_per_rb=1 if layout == 1 else 0, n_threads=8,
                        n_bearers=nb, grant_list_len=grants)
    _, dts = workload.tti_clock(T)
    seed = int(rng.integers(1, 1 << 30))
    refresh = int(rng.choice([1, 1, 7, 40]))
    if entry == "trace":   # trace replay: rows -1 (CQI 10) before the first report, some UEs on no trace at all
        n_tr, n_rows = 4, 7
        traces = rng.integers(1, 16, (n_tr, n_rows, R)).astype(np.uint8)
        if layout != 1:
            traces = np.repeat(traces[:, :, ::rbg], rbg, axis=2)
        ue_trace = rng.integers(-1, n_tr, (B, U)).astype(np.int32)
        rows = np.repeat(rng.integers(0, n_rows, T // 5 + 1), 5)[:T].astype(np.int32)
        rows[:int(rng.integers(0, 6))] = -1
        g.set_traces(traces, ue_trace)
    per = (B, U) if nb == 1 else (B, U, 2)
    feed = {"cqi": [], "draws": [], "active": [], "queue": [], "hol": []}
    want = []
    for t in range(T):
        if entry == "trace":
            cqi = ti.cqi_at(traces if layout == 1 else traces[:, :, ::rbg], ue_trace, int(rows[t]))
        else:
            cqi = workload.synth_cqi(seed, 0, B, t, 1, U, G, refresh)[0]
        dev_cqi = cqi
        if layout == 1 and entry != "trace":
            cqi = np.clip(np.repeat(cqi, rbg, axis=-1).astype(np.int64) + rng.integers(-1, 2, (B, U, R)), 1, 15).astype(np.uint8)
            dev_cqi = cqi
        elif layout == 2:
            dev_cqi = sched.pack_cqi(cqi)
        draws = workload.synth_rand_draws(seed, 0, B, t, 1, S, max(g.rand_stride, 2))[0]
        kw = {}
        if with_active:
            kw["active"] = (rng.random((B, U)) < 0.8).astype(np.uint8)
        if queue_aware:
            kind = rng.random(per)
            kw["queue"] = np.where(kind < 0.15, 0, np.where(kind < 0.6, rng.integers(20, 20000, per), 100000000)).astype(np.int32)
            kw["hol"] = np.where(rng.random(per) < 0.1, 0.0, rng.random(per) * 0.08)
            # a negative delay: "the bearer of the slice's priority is empty" of a caller that folds two bearers per UE.
            # Only where the ABI defines it (alpha without beta): in a slice whose metric carries the delay a negative
            # one makes metrics negative, which the reference cannot produce (it asserts when no user of a slice with
            # a quota qualifies, transport.cpp:609) -- found by the soak with seed 7, case 24.
            if nb == 1:
                gate_only = ((p[:, 0] != 0) & (p[:, 1] == 0))[u2s] if algo != 7 else np.zeros(U, dtype=bool)
                kw["hol"] = np.where((rng.random((B, U)) < 0.1) & gate_only[None, :], -1.0, kw["hol"])
        a = o.step(cqi, draws, dt=float(dts[t]), want_aux=True, **kw)
        if entry != "step":
            want.append(a)
            for k, v in (("cqi", dev_cqi), ("draws", draws)) + tuple(kw.items()):
                feed[k].append(v)
            continue
        b = g.step(dev_cqi, draws, dt=float(dts[t]), want_aux=True, **kw)
        for k in b:
            if not np.array_equal(a[k], b[k]):
                return f"case {case}: id {algo} S {S} U {U} layout {layout} queue {queue_aware} tti {t}: {k} differs"
    if entry != "step":
        kw = {k: np.stack(v) for k, v in feed.items() if v and k not in ("cqi", "draws")}
        if entry == "trace":
            b = g.run_traces_host(rows, np.stack(feed["draws"]), dts, want_aux=True, ttis_per_launch=tpl, **kw)
        else:
            b = g.run_host(np.stack(feed["cqi"]), np.stack(feed["draws"]), dts, want_aux=True, ttis_per_launch=tpl, **kw)
        for t in range(T):
            for k in b:
                if not np.array_equal(want[t][k], b[k][t]):
                    return (f"case {case}: id {algo} S {S} U {U} G {G} layout {layout} bearers {nb} queue {queue_aware} "
                            f"{entry} ttis_per_launch {tpl} tti {t}: {k} differs")
    sa, sb = o.get_state(), g.get_state()
    for k in ("avg_rate", "tx_bytes", "cum_bytes", "cum_rbs", "slice_offset", "nvs_ewma"):
        if k == "slice_offset" and algo not in (8, 9, 10, 101, 103):
            continue
        if k == "nvs_ewma" and algo not in (7, 11):
            continue
        if not np.array_equal(sa[k], sb[k]):
            return f"case {case}: id {algo} S {S} U {U} G {G} bearers {nb} {entry}: state {k} differs after {T} TTIs"
    g.close()
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--wide", action="store_true", help="also draw bands, two bearers, wide cells and multi-TTI entries")
    ap.add_argument("--limits", action="store_true", help="draw up to 64 slices, the bands and thousands of UEs")
    args = ap.parse_args()
    rng = np.random.default_rng(args.seed)
    t0, n, ttis = time.time(), 0, 0
    while time.time() - t0 < args.seconds:
        err = one_case(rng, n, wide=args.wide, limits=args.limits)
        if err:
            print("MISMATCH", err)
            return 1
        n += 1
    print(f"fuzz ok: {n} random configurations, no mismatch ({time.time() - t0:.0f} s, seed {args.seed})")
    return 0


if __name__ == "__main__":
    sys.exit(main())

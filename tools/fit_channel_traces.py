#!/usr/bin/env python3
"""Fit the example channel file tests/data/channel20x5_traces.json (rs_batch --channel, cfg20x5.json) to the committed
trace subset tests/golden/traces/trace_subset.npz: 127 cqi-traces-noise0 traces x their first 8 reports x 64 RBGs.

- level_counts: the histogram of the per-trace mean CQI, rounded to the nearest level;
- depth_cqi: the standard deviation of the CQI around each trace's own mean (within-trace spread);
- coherence_rbgs / coherence_reports: the integer coherence whose sinc(pi lag / coherence) is closest, in least squares,
  to the subset's autocorrelation over RBG lags 1..16 (each row's mean removed) and report lags 1..7 (each trace's
  mean removed).

The subset covers 320 ms, so the fit is indicative, not a validated channel model.

    python tools/fit_channel_traces.py            # writes tests/data/channel20x5_traces.json from the repository root
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "traces", "trace_subset.npz")
OUT = os.path.join(ROOT, "tests", "data", "channel20x5_traces.json")


def _corr(a, b):
    return float((a * b).mean() / np.sqrt((a * a).mean() * (b * b).mean()))


def _fit_coherence(corr):
    lags = np.arange(1, len(corr) + 1)
    err = {f: float(((np.sinc(lags / f) - np.asarray(corr)) ** 2).sum()) for f in range(1, 65)}
    return min(err, key=err.get)


def fit(rows):
    """rows [traces][reports][RBGs] -> the fields of one channel-file entry, and the statistics behind them."""
    r = rows.astype(np.float64)
    mean = r.mean(axis=(1, 2))
    level = np.clip(np.rint(mean), 1, 15).astype(int)
    counts = [int((level == v).sum()) for v in range(1, 16)]
    depth = float((r - mean[:, None, None]).std())
    d = r - r.mean(axis=2, keepdims=True)
    cf = [_corr(d[..., :-k], d[..., k:]) for k in range(1, 17)]
    t = r - mean[:, None, None]
    ct = [_corr(t[:, :-k], t[:, k:]) for k in range(1, r.shape[1])]
    entry = {"level_counts": counts, "depth_cqi": round(depth, 2), "coherence_rbgs": _fit_coherence(cf),
             "coherence_reports": _fit_coherence(ct)}
    return entry, {"rbg_corr": cf, "report_corr": ct, "trace_means": mean}


def main() -> int:
    z = np.load(FIX)
    entry, st = fit(z["rows"])
    note = (f"Fitted to a {z['rows'].shape[0]}-trace, {z['rows'].shape[1]}-report subset of cqi-traces-noise0 "
            "(tests/golden/traces/trace_subset.npz) by tools/fit_channel_traces.py; not a validated channel model. "
            "Levels: per-trace mean CQI; depth: within-trace standard deviation; coherences: least-squares sinc fits "
            f"to the RBG autocorrelation (lag 1: {st['rbg_corr'][0]:.2f}) and the report autocorrelation "
            f"(lag 1: {st['report_corr'][0]:.2f}). Reports every 40 TTIs, the reference's CQI_INTERVAL.")
    doc = {"note": note, "report_ttis": 40, "slices": [entry]}
    with open(OUT, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print(json.dumps(entry))
    return 0


if __name__ == "__main__":
    sys.exit(main())

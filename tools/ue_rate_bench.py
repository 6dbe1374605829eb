"""What the per-UE throughput histograms (rs_enable_ue_rate_hist, rs_batch --rate-window) cost.

Setup (one B200, synthetic CQI, id 9, 20 slices x 5 UEs, tests/data/cfg20x5.json, 1000 bins):
  (a) rs_close_ue_rate_window alone: device-event time of one close on the handle's stream, at 4096 and 65536 cells,
      one and two bearers per UE.  Each close follows a window of 8 TTIs (rs_run_device, not timed), so the samples
      spread over the bins as in a run (16-byte bins: a few per cent of the samples in the 64 bins counted in shared
      memory, the rest through the warp match to global memory); the line gives the median and the spread over
      --closes closes, and the bytes one close moves (the UE's nb counters and its snapshot read, the snapshot
      written) over its median time;
  (b) rs_batch --cells 4096 --ttis 2000 cell-TTIs/s without and with --rate-window 1000 --rate-bins 1000
      --rate-bin-bytes 10000, alternated over --rounds.
One JSON line per measurement, each with the card's name and power limit read in the same run.

    python tools/ue_rate_bench.py --out profiles/r09_ue_rate_hist.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import sched, workload  # noqa: E402

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg20x5.json")
BINS, TW = 1000, 8


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, limit = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": limit}


def batch(cells, ttis, window):
    args = [BIN, "--algo", "9", "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1"]
    if window:
        args += ["--rate-window", str(window), "--rate-bins", str(BINS), "--rate-bin-bytes", "10000"]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def close_time(cells, nb, warm, closes, bin_bytes=16):
    """(per-close device times in us, the histogram after the timed closes)."""
    import torch
    w, p, u2s = sched.load_slice_config(CFG)
    U = len(u2s)
    st = torch.cuda.Stream()
    g = sched.Scheduler(9, w, p, u2s, cells, cqi_per_rb=2, n_bearers=nb)
    g.set_stream(st.cuda_stream)
    d_cqi = torch.empty((TW, cells, U, 32), dtype=torch.uint8, device="cuda")
    d_r2 = torch.empty((TW, cells, 2), dtype=torch.int32, device="cuda")
    d_q = d_h = None
    if nb == 2:   # two backlogged bearers per UE: every run call takes queues (rs_set_queues)
        d_q = torch.full((TW, cells, U, 2), 100000000, dtype=torch.int32, device="cuda")
        d_h = torch.zeros((TW, cells, U, 2), dtype=torch.float64, device="cuda")
    _, dts = workload.tti_clock((warm + closes) * TW)
    g.enable_ue_rate_hist(BINS, bin_bytes)
    times = []
    for k in range(warm + closes):
        if k == warm:
            g.enable_ue_rate_hist(BINS, bin_bytes)   # zeroed: the histogram holds the timed closes only
        t0 = k * TW
        g.synth_cqi(1, 0, t0, TW, d_cqi.data_ptr())
        g.synth_rand2(1, 0, t0, TW, d_r2.data_ptr())
        g.run_device(TW, d_cqi.data_ptr(), cells * U * 32, d_r2.data_ptr(), dts[t0:t0 + TW], ttis_per_launch=TW,
                     d_queue=0 if d_q is None else d_q.data_ptr(), d_hol=0 if d_h is None else d_h.data_ptr())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        g.close_ue_rate_window()
        e1.record(st)
        e1.synchronize()
        if k >= warm:
            times.append(e0.elapsed_time(e1) * 1000.0)
    hist = g.get_ue_rate_hist()
    g.close()
    return np.array(times), hist


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ttis", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--closes", type=int, default=30)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    info = card()
    U = len(sched.load_slice_config(CFG)[2])
    lines = []
    for cells in (4096, 65536):
        for nb in (1, 2):
            t, hist = close_time(cells, nb, 5, a.closes)
            per_bin = hist.sum(axis=(0, 1))
            moved = cells * U * 8 * (nb + 2)
            med = float(np.median(t))
            lines.append(dict(info, arm="close_ue_rate_window", cells=cells, ues=U, bearers=nb, bins=BINS, bin_bytes=16,
                              closes=a.closes, close_us_median=round(med, 2), close_us_min=round(float(t.min()), 2),
                              close_us_max=round(float(t.max()), 2), bytes_per_close=moved,
                              gb_per_s_at_median=round(moved / (med * 1e-6) / 1e9, 1),
                              samples=int(per_bin.sum()), samples_bins_0_63=int(per_bin[:64].sum()),
                              samples_bins_64_998=int(per_bin[64:-1].sum()), samples_last_bin=int(per_bin[-1])))
            print(json.dumps(lines[-1]), flush=True)
    for r in range(a.rounds):
        for arm, window in (("rs_batch", 0), ("rs_batch_rate_window_1000_bins_1000", 1000)):
            res = batch(4096, a.ttis, window)
            line = dict(info, arm=arm, round=r, cells=4096, ttis=a.ttis, cell_ttis_per_s=res["cell_ttis_per_s"])
            if window:
                line.update(ue_rate_samples=sum(res["ue_rate_samples"]), ue_rate_p5=res["ue_rate_p5"][:3],
                            ue_rate_p50=res["ue_rate_p50"][:3], ue_rate_p95=res["ue_rate_p95"][:3])
            lines.append(line)
            print(json.dumps(line), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

"""What the head-of-line delay histograms (rs_enable_hol_hist, rs_batch --hol-bins) cost.

Setup (one B200, synthetic CQI, id 9, 4096 cells x 20 slices x 5 UEs): tests/data/cfg20x5_ab.json with
tests/data/traffic20x5_video_voip.json, 64 records per bearer, 1000 1-TTI bins.
  (a) the reducer: a closed loop of 16-TTI rs_run_device calls (as rs_batch runs it) under torch.profiler; the mean
      device time of rs_hol_hist_kernel per call against that of the TTI kernel it follows;
  (b) rs_batch cell-TTIs/s without and with --hol-bins 1000, alternated over --rounds.
One JSON line per measurement, each with the card's name and power limit read in the same run.

    python tools/hol_hist_bench.py --out profiles/r08_hol_hist.jsonl
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
CFG = os.path.join(ROOT, "tests", "data", "cfg20x5_ab.json")
TRAFFIC = os.path.join(ROOT, "tests", "data", "traffic20x5_video_voip.json")
K, BINS, TB = 64, 1000, 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, limit = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": limit}


def batch(cells, ttis, bins):
    args = [BIN, "--algo", "9", "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1", "--buffers",
            str(K), "--traffic", TRAFFIC]
    if bins:
        args += ["--hol-bins", str(bins)]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def reducer_time(cells, warm_calls, calls):
    """(us of rs_hol_hist_kernel per call, us of the TTI kernel per call, kernels seen, the histogram's samples)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    w, p, u2s = sched.load_slice_config(CFG)
    nb, bl, src = sched.load_traffic(TRAFFIC, CFG)
    U = len(u2s)
    g = sched.Scheduler(9, w, p, u2s, cells, cqi_per_rb=2, n_bearers=nb)
    g.enable_buffers(K, np.broadcast_to(bl, (cells,) + bl.shape))
    g.set_sources(src)
    g.enable_hol_hist(BINS)
    n = warm_calls + calls
    now, dts = workload.tti_clock(n * TB)
    d_arr = torch.empty((TB, cells, U, nb), dtype=torch.int32, device="cuda")
    d_cqi = torch.empty((TB, cells, U, 32), dtype=torch.uint8, device="cuda")
    d_r2 = torch.empty((TB, cells, 2), dtype=torch.int32, device="cuda")

    def call(k):
        t0 = k * TB
        g.synth_traffic(1, 0, t0, TB, d_arr.data_ptr())
        g.synth_cqi(1, 0, t0, TB, d_cqi.data_ptr())
        g.synth_rand2(1, 0, t0, TB, d_r2.data_ptr())
        g.run_device(TB, d_cqi.data_ptr(), cells * U * 32, d_r2.data_ptr(), dts[t0:], d_arrivals=d_arr.data_ptr(),
                     now=now[t0:t0 + TB], ttis_per_launch=TB)

    for k in range(warm_calls):
        call(k)
    g.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(warm_calls, n):
            call(k)
        g.sync()
    hist = g.get_hol_hist()
    g.close()
    red = tti = 0.0
    seen = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "rs_hol_hist_kernel" in e.key:
            red += t
            seen["reducer"] = seen.get("reducer", 0) + e.count
        elif "rs_tti_kernel" in e.key:
            tti += t
            seen["tti_kernel"] = seen.get("tti_kernel", 0) + e.count
    return red / calls, tti / calls, seen, hist


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=4096)
    ap.add_argument("--ttis", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=60)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    info = card()
    lines = []
    red, tti, seen, hist = reducer_time(a.cells, 20, a.calls)
    lines.append(dict(info, arm="reducer_per_16_tti_call", cells=a.cells, bins=BINS, calls=a.calls, kernels=seen,
                      hol_hist_us=round(red, 2), tti_kernel_us=round(tti, 2), share=round(red / tti, 5),
                      served_samples=int(hist[:, 0].sum()), waiting_samples=int(hist[:, 1].sum()),
                      last_bin_waiting=int(hist[:, 1, :, -1].sum())))
    print(json.dumps(lines[-1]), flush=True)
    for r in range(a.rounds):
        for arm, bins in (("rs_batch_buffers_64", 0), ("rs_batch_buffers_64_hol_bins_1000", BINS)):
            res = batch(a.cells, a.ttis, bins)
            line = dict(info, arm=arm, round=r, cells=a.cells, ttis=a.ttis, cell_ttis_per_s=res["cell_ttis_per_s"])
            if bins:
                line.update(hol_served=sum(res["hol_served"]), hol_waiting=sum(res["hol_waiting"]),
                            hol_waiting_p99=res["hol_waiting_p99"])
            lines.append(line)
            print(json.dumps(line), flush=True)
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

"""What the closed loop costs the C++ batch program, and what the per-slice buffer totals cost.

Arms, alternated over --rounds (one B200 process each, synthetic CQI, id 9, 4096 cells x 20 slices x 5 UEs):
  (a) rs_batch --config tests/data/cfg20x5_ab.json                 every bearer backlogged (no flag)
  (b) the same with --buffers 64 --traffic tests/data/traffic20x5_ab.json: the even slices are alpha/beta slices fed
      1500-byte packets at 0.6 or 0.15 per TTI (as tools/buffer_bench.py), the odd ones stay backlogged
and the time of one rs_buffer_stats_device call on a handle of that size after a closed loop (CUDA events around
--reps back-to-back calls).  One JSON line per measurement, each with the card's name and power limit.

    python tools/rs_batch_buffers_bench.py --out profiles/r05_rs_batch_closed_loop.jsonl
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
TRAFFIC = os.path.join(ROOT, "tests", "data", "traffic20x5_ab.json")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, limit = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": limit}


def batch(cells, ttis, buffers):
    args = [BIN, "--algo", "9", "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1"]
    if buffers:
        args += ["--buffers", str(buffers), "--traffic", TRAFFIC]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def stats_time(cells, ttis, reps):
    import torch
    w, p, u2s = sched.load_slice_config(CFG)
    nb, bl, pkt, q16 = sched.load_traffic_config(TRAFFIC, CFG)
    S, U = len(w), len(u2s)
    g = sched.Scheduler(9, w, p, u2s, cells, n_bearers=nb)
    g.enable_buffers(64, np.broadcast_to(bl[:, 0], (cells, U)))
    now, dts = workload.tti_clock(ttis)
    d_arr = torch.empty((ttis, cells, U), dtype=torch.int32, device="cuda")
    d_cqi = torch.empty((ttis, cells, U, 64), dtype=torch.uint8, device="cuda")
    d_r2 = torch.empty((ttis, cells, 2), dtype=torch.int32, device="cuda")
    g.synth_arrivals(1, 0, 0, ttis, pkt, q16, d_arr.data_ptr())
    g.synth_cqi(1, 0, 0, ttis, d_cqi.data_ptr())
    g.synth_rand2(1, 0, 0, ttis, d_r2.data_ptr())
    g.run_device(ttis, d_cqi.data_ptr(), cells * U * 64, d_r2.data_ptr(), dts, d_arrivals=d_arr.data_ptr(), now=now,
                 ttis_per_launch=16)
    d = torch.empty(3 * S, dtype=torch.int64, device="cuda")
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    for _ in range(10):
        g.buffer_stats_device(d.data_ptr())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.buffer_stats_device(d.data_ptr())
    e1.record()
    e1.synchronize()
    st = g.get_buffer_stats()
    g.close()
    return e0.elapsed_time(e1) * 1e3 / reps, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=4096)
    ap.add_argument("--ttis", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    info = card()
    lines = []
    for r in range(a.rounds):
        for arm, k in (("a_backlogged", 0), ("b_buffers_64", 64)):
            res = batch(a.cells, a.ttis, k)
            line = dict(info, arm=arm, round=r, cells=a.cells, ttis=a.ttis, cell_ttis_per_s=res["cell_ttis_per_s"])
            if k:
                line.update(queued_bytes=sum(res["queued_bytes"]), dropped_bytes=sum(res["dropped_bytes"]),
                            records=sum(res["records"]))
            lines.append(line)
            print(json.dumps(line), flush=True)
    us, st = stats_time(a.cells, 64, a.reps)
    line = dict(info, arm="rs_buffer_stats_device", cells=a.cells, bearers=a.cells * 100, reps=a.reps, us_per_call=round(us, 2),
                queued_bytes=int(st[0].sum()), records=int(st[2].sum()))
    lines.append(line)
    print(json.dumps(line), flush=True)
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

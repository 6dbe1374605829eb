"""What the per-UE throughput over active time (UPT) histograms (rs_enable_ue_upt_hist, rs_batch --upt-bin-bytes) cost,
and what they show that the window histograms do not.

Setup (one B200, synthetic CQI, id 9, 20 slices x 5 UEs): tests/data/cfg20x5_ab.json with
tests/data/traffic20x5_video_voip.json, 64 records per bearer, 1000 bins.
  (a) the active-count kernel: a closed loop of 16-TTI rs_run_device calls (as rs_batch runs it) at 4096 cells under
      torch.profiler; the mean device time of rs_ue_active_kernel per call against that of the TTI kernel it follows,
      and the bytes it reads (the queues the 16 TTIs showed) over its time;
  (b) one close: device-event time of rs_close_ue_rate_window with UPT off and on, at 4096 and 65536 cells, each close
      after a 16-TTI window (not timed); the line gives the median and the spread over --closes closes;
  (c) rs_batch --cells 4096 --ttis 2000 --rate-window 1000 --rate-bins 1000 --rate-bin-bytes 10000 cell-TTIs/s
      without and with --upt-bin-bytes 100, alternated over --rounds;
  (d) the same traffic under ids 8 and 9 (rs_batch --cells 1024 --ttis 2000, 1000-TTI windows of 100-byte bins, UPT in
      20-byte-per-TTI bins): the 5th percentiles of both histograms per slice.
One JSON line per measurement, each with the card's name and power limit read in the same run.

    python tools/upt_bench.py --out profiles/r11_ue_upt_hist.jsonl
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


def batch(algo, cells, ttis, *extra):
    args = [BIN, "--algo", str(algo), "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1",
            "--buffers", str(K), "--traffic", TRAFFIC, *[str(x) for x in extra]]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


class Loop:
    """A buffered id-9 handle of `cells` cells fed by its device sources, run in 16-TTI rs_run_device calls."""

    def __init__(self, cells, upt):
        import torch
        w, p, u2s = sched.load_slice_config(CFG)
        nb, bl, src = sched.load_traffic(TRAFFIC, CFG)
        self.U, self.cells, self.nb = len(u2s), cells, nb
        self.g = sched.Scheduler(9, w, p, u2s, cells, cqi_per_rb=2, n_bearers=nb)
        self.g.enable_buffers(K, np.broadcast_to(bl, (cells,) + bl.shape))
        self.g.set_sources(src)
        self.g.enable_ue_rate_hist(BINS, 10000)
        if upt:
            self.g.enable_ue_upt_hist(BINS, 100)
        self.d_arr = torch.empty((TB, cells, self.U, nb), dtype=torch.int32, device="cuda")
        self.d_cqi = torch.empty((TB, cells, self.U, 32), dtype=torch.uint8, device="cuda")
        self.d_r2 = torch.empty((TB, cells, 2), dtype=torch.int32, device="cuda")
        self.now, self.dts = workload.tti_clock(4000 * TB)

    def call(self, k):
        g, t0 = self.g, k * TB
        g.synth_traffic(1, 0, t0, TB, self.d_arr.data_ptr())
        g.synth_cqi(1, 0, t0, TB, self.d_cqi.data_ptr())
        g.synth_rand2(1, 0, t0, TB, self.d_r2.data_ptr())
        g.run_device(TB, self.d_cqi.data_ptr(), self.cells * self.U * 32, self.d_r2.data_ptr(), self.dts[t0:],
                     d_arrivals=self.d_arr.data_ptr(), now=self.now[t0:t0 + TB], ttis_per_launch=TB)


def active_time(cells, warm_calls, calls):
    """(us of rs_ue_active_kernel per call, us of the TTI kernel per call, kernels seen)."""
    from torch.profiler import ProfilerActivity, profile
    lp = Loop(cells, True)
    for k in range(warm_calls):
        lp.call(k)
    lp.g.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(warm_calls, warm_calls + calls):
            lp.call(k)
        lp.g.sync()
    lp.g.close()
    act = tti = 0.0
    seen = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "rs_ue_active_kernel" in e.key:
            act += t
            seen["active"] = seen.get("active", 0) + e.count
        elif "rs_tti_kernel" in e.key:
            tti += t
            seen["tti_kernel"] = seen.get("tti_kernel", 0) + e.count
    return act / calls, tti / calls, seen


def close_time(cells, upt, warm, closes):
    """(per-close device times in us, UPT samples or None)."""
    import torch
    lp = Loop(cells, upt)
    st = torch.cuda.Stream()
    lp.g.set_stream(st.cuda_stream)
    times = []
    for k in range(warm + closes):
        lp.call(k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        lp.g.close_ue_rate_window()
        e1.record(st)
        e1.synchronize()
        if k >= warm:
            times.append(e0.elapsed_time(e1) * 1000.0)
    samples = int(lp.g.get_ue_upt_hist().sum()) if upt else None
    lp.g.close()
    return np.array(times), samples


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ttis", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=60)
    ap.add_argument("--closes", type=int, default=30)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    info = card()
    lines = []

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)

    cells = 4096
    act, tti, seen = active_time(cells, 20, a.calls)
    U = len(sched.load_slice_config(CFG)[2])
    read = TB * cells * U * 4   # the shown queues of one call, one bearer per UE
    emit(dict(info, arm="active_kernel_per_16_tti_call", cells=cells, calls=a.calls, kernels=seen,
              active_us=round(act, 2), tti_kernel_us=round(tti, 2), share=round(act / tti, 5), bytes_read=read,
              gb_per_s=round(read / (act * 1e-6) / 1e9, 1)))
    for c in (4096, 65536):
        for upt in (False, True):
            t, samples = close_time(c, upt, 5, a.closes)
            emit(dict(info, arm="close_ue_rate_window_upt_" + ("on" if upt else "off"), cells=c, closes=a.closes,
                      close_us_median=round(float(np.median(t)), 2), close_us_min=round(float(t.min()), 2),
                      close_us_max=round(float(t.max()), 2), upt_samples=samples))
    rate = ["--rate-window", 1000, "--rate-bins", BINS, "--rate-bin-bytes", 10000]
    for r in range(a.rounds):
        for arm, extra in (("rs_batch_rate_window_1000", []), ("rs_batch_rate_window_1000_upt_100", ["--upt-bin-bytes", 100])):
            res = batch(9, cells, a.ttis, *rate, *extra)
            line = dict(info, arm=arm, round=r, cells=cells, ttis=a.ttis, cell_ttis_per_s=res["cell_ttis_per_s"])
            if extra:
                line.update(upt_samples=sum(res["upt_samples"]), upt_p5=res["upt_p5"][:4])
            emit(line)
    for algo in (8, 9):
        res = batch(algo, 1024, a.ttis, "--rate-window", 1000, "--rate-bins", 4000, "--rate-bin-bytes", 100,
                    "--upt-bin-bytes", 20)
        emit(dict(info, arm="video_voip_p5", algo=algo, cells=1024, ttis=a.ttis, rate_bin_bytes=100, upt_bin_bytes=20,
                  ue_rate_p5=res["ue_rate_p5"], upt_p5=res["upt_p5"], upt_p50=res["upt_p50"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

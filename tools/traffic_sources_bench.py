"""What drawing traffic on the device costs, and what periodic / on-off traffic does to the closed loop's rate.

One B200 process, id 9, 4096 cells x 20 slices x 5 UEs (tests/data/cfg20x5_ab.json), one bearer per UE:
  (a) one 16-TTI chunk of arrivals, CUDA events around --reps back-to-back calls of each generator arm, arms alternated
      over --rounds: rs_synth_arrivals with the rate file tests/data/traffic20x5_ab.json; rs_synth_traffic with the same
      file as RATE sources (the same output); rs_synth_traffic with tests/data/traffic20x5_video_voip.json (periodic
      frames and on-off sources on the alpha/beta slices).  Each chunk writes 16 x 409 600 int32 = 26.2 MB, more than
      the L2 holds, so every call writes HBM;
  (b) rs_batch --buffers 64 closed-loop rates with each traffic file, arms alternated over --rounds.  rs_batch times its
      scheduling calls only, so these rates show what the traffic does to the TTI kernel, not the generator's cost.
One JSON line per measurement, each with the card's name and power limit.

    python tools/traffic_sources_bench.py --out profiles/r06_traffic_sources.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import sched  # noqa: E402

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg20x5_ab.json")
RATE = os.path.join(ROOT, "tests", "data", "traffic20x5_ab.json")
VIDEO_VOIP = os.path.join(ROOT, "tests", "data", "traffic20x5_video_voip.json")
CHUNK = 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, limit = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": limit}


def generator_times(cells, reps, rounds):
    """{arm: [(device us per 16-TTI call, host us to enqueue one), one per round]}.  When the two are close, the calls
    were enqueued no faster than the device ran them: the device time is then an upper bound on the kernel's."""
    import torch
    w, p, u2s = sched.load_slice_config(CFG)
    _, _, pkt, q16 = sched.load_traffic_config(RATE, CFG)
    _, _, rate_src = sched.load_traffic(RATE, CFG)
    _, _, vv_src = sched.load_traffic(VIDEO_VOIP, CFG)
    gens = {}
    for arm, src in (("synth_arrivals_rate", None), ("synth_traffic_rate", rate_src), ("synth_traffic_video_voip", vv_src)):
        g = sched.Scheduler(9, w, p, u2s, cells)
        g.set_stream(torch.cuda.current_stream().cuda_stream)
        if src is not None:
            g.set_sources(src)
        gens[arm] = [g, 0]   # handle, next TTI
    out = torch.empty((CHUNK, cells, len(u2s)), dtype=torch.int32, device="cuda")

    def call(arm):
        g, t = gens[arm]
        if arm == "synth_arrivals_rate":
            g.synth_arrivals(1, 0, t, CHUNK, pkt, q16, out.data_ptr())
        else:
            g.synth_traffic(1, 0, t, CHUNK, out.data_ptr())
        gens[arm][1] = t + CHUNK

    times = {arm: [] for arm in gens}
    for arm in gens:   # warm-up
        for _ in range(20):
            call(arm)
    for _ in range(rounds):
        for arm in gens:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            h0 = time.perf_counter()
            for _ in range(reps):
                call(arm)
            h1 = time.perf_counter()
            e1.record()
            e1.synchronize()
            times[arm].append((e0.elapsed_time(e1) * 1e3 / reps, (h1 - h0) * 1e6 / reps))
    for g, _ in gens.values():
        g.close()
    return times


def batch(cells, ttis, traffic):
    args = [BIN, "--algo", "9", "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1", "--buffers", "64",
            "--traffic", traffic]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


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

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)

    bearers = a.cells * 100
    for arm, us in generator_times(a.cells, a.reps, a.rounds).items():
        for r, (x, host) in enumerate(us):
            emit(dict(info, arm=arm, round=r, cells=a.cells, bearers=bearers, ttis_per_call=CHUNK, reps=a.reps,
                      us_per_call=round(x, 2), host_enqueue_us_per_call=round(host, 2),
                      hbm_write_gb_per_s=round(CHUNK * bearers * 4 / (x * 1e-6) / 1e9, 1)))
    for r in range(a.rounds):
        for arm, traffic in (("rs_batch_rate", RATE), ("rs_batch_video_voip", VIDEO_VOIP)):
            res = batch(a.cells, a.ttis, traffic)
            emit(dict(info, arm=arm, round=r, cells=a.cells, ttis=a.ttis, cell_ttis_per_s=res["cell_ttis_per_s"],
                      ms_per_16_tti_chunk=round(CHUNK * a.cells / res["cell_ttis_per_s"] * 1e3, 3),
                      queued_bytes=sum(res["queued_bytes"]), dropped_bytes=sum(res["dropped_bytes"]),
                      records=sum(res["records"])))
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

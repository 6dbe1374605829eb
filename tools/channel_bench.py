"""What drawing the synthetic channel on the device costs, next to rs_synth_cqi and next to a TTI.

One B200 process, 4096 cells x 20 slices x 5 UEs x 64 RBGs (tests/data/cfg20x5.json):
  (a) generator time per slab: CUDA events around --reps back-to-back calls of each arm, arms alternated over --rounds:
      rs_synth_cqi and rs_synth_channel with tests/data/channel20x5_traces.json (FADING on every slice), each in layout 0
      (u8 per RBG, 26.2 MB per slab) and layout 2 (4-bit packed, 13.1 MB), in calls of 1 slab (what rs_batch draws per
      chunk at report_ttis 40) and of 16 slabs (report_ttis 1).  The host time to enqueue a call is reported next to
      the device time: when the two are close the calls are launch-bound and the device time is an upper bound.  The
      floor is the bytes written per slab over the data sheet's 7.7 TB/s;
  (b) rs_batch rates for id 9 over --ttis TTIs, arms alternated over --rounds: without --channel, an all-IID file at
      report_ttis 1, the example file at report_ttis 1 and at 40.  rs_batch times its scheduling calls only, so the
      rates give the TTI's time without the generator.
One JSON line per measurement, each with the card's name and power limit.

    python tools/channel_bench.py --out profiles/r07_synth_channel.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import sched  # noqa: E402

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
CFG = os.path.join(ROOT, "tests", "data", "cfg20x5.json")
EXAMPLE = os.path.join(ROOT, "tests", "data", "channel20x5_traces.json")
HBM_BYTES_PER_S = 7.7e12   # NVIDIA HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, limit = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": limit}


def generator_times(cells, reps, rounds):
    """{(arm, layout, slabs per call): [(device us per slab, host us to enqueue one call), one per round]}."""
    import torch
    w, p, u2s = sched.load_slice_config(CFG)
    _, chans = sched.load_channel(EXAMPLE, CFG)
    stream = torch.cuda.Stream()   # a stream of its own: the events below are recorded on the stream the calls run on
    handles = {}
    for layout in (0, 2):
        g = sched.Scheduler(9, w, p, u2s, cells, cqi_per_rb=layout)
        g.set_stream(stream.cuda_stream)
        g.set_channels(chans)
        handles[layout] = g
    out = torch.empty(16 * cells * len(u2s) * 64, dtype=torch.uint8, device="cuda")
    arms = [(arm, layout, n) for n in (1, 16) for layout in (0, 2) for arm in ("synth_cqi", "synth_channel")]
    epoch = {a: 0 for a in arms}

    def call(a):
        arm, layout, n = a
        getattr(handles[layout], arm)(1, 0, epoch[a], n, out.data_ptr())
        epoch[a] += n

    times = {a: [] for a in arms}
    for a in arms:   # warm-up
        for _ in range(10):
            call(a)
    stream.synchronize()
    for _ in range(rounds):
        for a in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            h0 = time.perf_counter()
            for _ in range(reps):
                call(a)
            h1 = time.perf_counter()
            e1.record(stream)
            e1.synchronize()
            times[a].append((e0.elapsed_time(e1) * 1e3 / reps / a[2], (h1 - h0) * 1e6 / reps))
    for g in handles.values():
        g.close()
    return times


def batch(cells, ttis, channel):
    args = [BIN, "--algo", "9", "--config", CFG, "--cells", str(cells), "--ttis", str(ttis), "--seed", "1"]
    if channel:
        args += ["--channel", channel]
    r = subprocess.run(args, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=4096)
    ap.add_argument("--ttis", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    info = card()
    lines = []

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)

    rows = a.cells * 100
    for (arm, layout, n), us in generator_times(a.cells, a.reps, a.rounds).items():
        slab_bytes = rows * (64 if layout == 0 else 32)
        for r, (x, host) in enumerate(us):
            emit(dict(info, arm=arm, layout=layout, slabs_per_call=n, round=r, cells=a.cells, ues=100, rbgs=64,
                      reps=a.reps, us_per_slab=round(x, 2), host_enqueue_us_per_call=round(host, 2),
                      us_per_call=round(x * n, 2), bytes_per_slab=slab_bytes,
                      floor_us_per_slab=round(slab_bytes / HBM_BYTES_PER_S * 1e6, 2)))
    with open(EXAMPLE) as f:
        example = json.load(f)
    with tempfile.TemporaryDirectory() as tmp:
        files = {"no_flag": None}
        for name, doc in (("all_iid_r1", {"report_ttis": 1, "slices": [{"iid": 1}]}),
                          ("example_r1", dict(example, report_ttis=1)), ("example_r40", example)):
            files[name] = os.path.join(tmp, name + ".json")
            with open(files[name], "w") as f:
                json.dump(doc, f)
        for r in range(a.rounds):
            for arm, path in files.items():
                res = batch(a.cells, a.ttis, path)
                emit(dict(info, arm="rs_batch_" + arm, round=r, cells=a.cells, ttis=a.ttis,
                          cell_ttis_per_s=res["cell_ttis_per_s"],
                          us_per_tti=round(a.cells / res["cell_ttis_per_s"] * 1e6, 2),
                          slice_bytes=sum(res["slice_bytes"])))
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

"""Cost of the device-kept per-bearer buffers (rs_enable_buffers), one JSON line per measured arm and round.

Batch: 4096 cells x 20 slices x 5 UEs, 64 RBGs, RadioSaber (id 9), synthetic CQI and rand() draws resident in HBM.
Slices 0, 2, .. weigh the head-of-line delay in (alpha = beta = 1) and get synthetic arrivals (rs_synth_arrivals: 1500 B
packets, 0.15 or 0.6 per TTI, so some queues drain and others build up to the 64-record limit); slices 1, 3, .. are
backlogged.  The arms run one after the other, round after round (--rounds), so that slow drift hits them all alike:

  closed     (a) the closed loop on the device: rs_set_traffic + rs_run_device, steps of 96 TTIs in launches of 16
  host       (b) the same loop driven from the host one TTI per call: rs_set_queues + rs_step + rs_get_state per TTI,
                 replaying the queue sizes and delays (a) showed (the host's own FIFO bookkeeping is not counted)
  replay     (c) (a)'s queue_out / hol_out replayed through rs_set_queues (device pointers) in the same launches: the
                 difference to (a) is the cost of the FIFO bookkeeping in the kernel
  backlogged (d) the same cells with every bearer backlogged (no queue state at all)

Timing: CUDA events on the launching stream around `--steps` steps after `--warmup` steps, cross-checked against the host
clock; (b) times steps of 16 TTIs.  The card's name and power limit are read in the same run.

    python tools/buffer_bench.py --out profiles/r04_closed_loop_buffers.jsonl [--rounds 3] [--steps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import sched, workload  # noqa: E402

S, UPS, G, B, SEED = 20, 5, 64, 4096, 1
U = S * UPS
TT, TPL, TT_HOST, K = 96, 16, 16, 64


def config():
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    p[0::2, :2] = 1
    u2s = np.repeat(np.arange(S), UPS).astype(np.int32)
    pkt = np.where(np.arange(S) % 2 == 0, 1500, 0).astype(np.int32)
    q16 = np.where(np.arange(S) % 4 == 0, int(0.6 * 65536), int(0.15 * 65536)).astype(np.int32)
    backlogged = np.broadcast_to((np.arange(S) % 2 == 1)[u2s], (B, U))
    return w, p, u2s, pkt, q16, backlogged


class Bench:
    def __init__(self, torch, dev, stream):
        self.torch, self.dev, self.stream = torch, dev, stream
        w, p, u2s, self.pkt, self.q16, self.backlogged = config()
        self.g = {}
        for arm in ("closed", "host", "replay", "backlogged"):
            g = sched.Scheduler(9, w, p, u2s, B, device=dev.index)
            g.set_stream(stream.cuda_stream)
            self.g[arm] = g
        g = self.g["closed"]
        e = torch.empty
        self.cqi = e((TT, B, U, G), dtype=torch.uint8, device=dev)
        self.r2 = e((TT, B, 2), dtype=torch.int32, device=dev)
        self.arr = e((TT, B, U), dtype=torch.int32, device=dev)
        self.qrec = e((TT, B, U), dtype=torch.int32, device=dev)
        self.hrec = e((TT, B, U), dtype=torch.float64, device=dev)
        g.synth_cqi(SEED, 0, 0, TT, self.cqi.data_ptr())
        g.synth_rand2(SEED, 0, 0, TT, self.r2.data_ptr())
        g.synth_arrivals(SEED, 0, 0, TT, self.pkt, self.q16, self.arr.data_ptr())
        out = {"rbg_to_ue": e((TT, B, G), dtype=torch.int16, device=dev), "tbs_bits": e((TT, B, U), dtype=torch.int32, device=dev),
               "mcs": e((TT, B, U), dtype=torch.uint8, device=dev)}
        self.out, self.ptrs = out, {k: v.data_ptr() for k, v in out.items()}
        self.now_ttis = 0
        _, self.dts = workload.tti_clock(TT)
        # (a) once from empty buffers, recording what the TTIs showed: (c) and (b) replay it
        g.enable_buffers(K, self.backlogged)
        self.closed_step(record=True)
        torch.cuda.synchronize(dev)
        q = self.qrec.cpu().numpy()
        buf = ~self.backlogged
        self.shown = {"drained": bool(((q[1:] == 0) & (q[:-1] > 0) & buf).any()), "max_queue": int(q[:, buf].max()),
                      "dropped_bytes": int(g.get_buffers()["dropped"].sum())}
        self.host_in = (self.cqi[:TT_HOST].cpu().numpy(), self.r2[:TT_HOST].cpu().numpy(), q[:TT_HOST].copy(),
                        self.hrec[:TT_HOST].cpu().numpy())

    def closed_step(self, record=False):
        now = 0.1 + 0.001 * np.arange(self.now_ttis, self.now_ttis + TT)
        self.now_ttis += TT
        self.g["closed"].run_device(TT, self.cqi.data_ptr(), B * U * G, self.r2.data_ptr(), self.dts, self.ptrs,
                                    ttis_per_launch=TPL, d_arrivals=self.arr.data_ptr(), now=now, arrival_time=now,
                                    d_queue_out=self.qrec.data_ptr() if record else 0,
                                    d_hol_out=self.hrec.data_ptr() if record else 0)

    def step(self, arm):
        if arm == "closed":
            self.closed_step()
        elif arm == "replay":
            self.g[arm].run_device(TT, self.cqi.data_ptr(), B * U * G, self.r2.data_ptr(), self.dts, self.ptrs,
                                   ttis_per_launch=TPL, d_queue=self.qrec.data_ptr(), d_hol=self.hrec.data_ptr())
        elif arm == "backlogged":
            self.g[arm].run_device(TT, self.cqi.data_ptr(), B * U * G, self.r2.data_ptr(), self.dts, self.ptrs,
                                   ttis_per_launch=TPL)
        else:
            g = self.g[arm]
            cqi, r2, q, h = self.host_in
            for t in range(TT_HOST):
                g.step(cqi[t], r2[t], dt=float(self.dts[t]), queue=q[t], hol=h[t])
                g.get_state()

    def ttis(self, arm):
        return TT_HOST if arm == "host" else TT


def time_arm(torch, bench, arm, steps, warmup):
    for _ in range(warmup):
        bench.step(arm)
    torch.cuda.synchronize(bench.dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    e0.record(bench.stream)
    for _ in range(steps):
        bench.step(arm)
    e1.record(bench.stream)
    torch.cuda.synchronize(bench.dev)
    wall_ms = (time.perf_counter() - wall0) * 1e3
    ms = e0.elapsed_time(e1)
    if not (0.8 * wall_ms <= ms <= 1.02 * wall_ms + 0.5):
        raise RuntimeError(f"{arm}: events {ms:.3f} ms disagree with the host clock {wall_ms:.3f} ms")
    return ms, wall_ms


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--arms", default="closed,host,replay,backlogged")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("buffer_bench: needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    props = torch.cuda.get_device_properties(dev)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    bench = Bench(torch, dev, stream)
    names = args.arms.split(",")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in range(args.rounds):
            for n in names:
                ms, wall = time_arm(torch, bench, n, args.steps, args.warmup)
                tt = bench.ttis(n)
                line = {"arm": n, "round": r, "cells": B, "slices": S, "ues": U, "algo": 9, "max_records": K,
                        "ttis_per_step": tt, "ttis_per_launch": 1 if n == "host" else TPL, "steps": args.steps,
                        "warmup_steps": args.warmup, "ms": round(ms, 3), "wall_ms": round(wall, 3),
                        "cell_ttis_per_s": B * tt * args.steps / (ms * 1e-3), **bench.shown,
                        "gpu": props.name, "power_limit": power}
                f.write(json.dumps(line) + "\n")
                f.flush()
                print(json.dumps(line), flush=True)
    for g in bench.g.values():
        g.close()


if __name__ == "__main__":
    main()

"""Throughput of slice profiles (rs_create_profiles) on the headline workload, one JSON line per measured arm.

Batch: 4096 cells x 20 slices x 5 UEs, 64 RBGs, RadioSaber (id 9), synthetic CQI (one byte per RBG) and rand() draws
resident in HBM.  Timing as in bench.py: steps of 96 TTIs in launches of 16, >= 224 warm-up TTIs per arm, CUDA events
on the launching stream, cross-checked against the host clock around the same synchronised region.  The arms run one
after the other, round after round (--rounds), so that slow drift of the machine hits them all alike:

  create        rs_create (the one-configuration handle bench.py times)
  p1            rs_create_profiles with one profile
  p20           20 weight / parameter profiles of the 20 x 5 cell (the compile-time-shape kernel)
  p4096         one profile per cell
  p20_mixed     20 profiles that also differ in UEs per slice (the general kernel)
  one_handle64  64 profiles (P = 20 style settings) x 64 cells of each in ONE handle of 4096 cells
  handles64     the same 64 settings as 64 handles of 64 cells, run one after another

    python tools/profile_bench.py --out profiles/r03_slice_profiles.jsonl [--rounds 3] [--steps 10]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import sched, workload  # noqa: E402

S, UPS, G, B, SEED = 20, 5, 64, 4096, 1
U = S * UPS
TT, TPL = 96, 16


def _weights_params(rng):
    w = rng.dirichlet(np.ones(S))
    p = np.zeros((S, 4), dtype=np.int32)
    p[:, 2] = rng.choice([0, 1, 2], S)
    p[:, 3] = rng.integers(0, 2, S)
    return w, p


def _headline():
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    return w, p, np.repeat(np.arange(S), UPS).astype(np.int32)


def _mixed_u2s(rng):
    ups = np.full(S, UPS)
    for _ in range(30):   # move UEs between slices, every slice keeps at least one
        a, b = rng.integers(0, S, 2)
        if ups[a] > 1:
            ups[a] -= 1
            ups[b] += 1
    return np.repeat(np.arange(S), ups).astype(np.int32)


def arms(rng):
    """{name: [(profiles, cell_profile or None, n_cells), ...]} -- one entry per handle of the arm."""
    w0, p0, u0 = _headline()
    prof20 = [_weights_params(rng) + (u0,) for _ in range(20)]
    mixed = [_weights_params(rng) + (_mixed_u2s(rng),) for _ in range(20)]
    prof4096 = [_weights_params(rng) + (u0,) for _ in range(B)]
    prof64 = [_weights_params(rng) + (u0,) for _ in range(64)]
    scatter = rng.permutation(np.arange(B) % 20)
    return {
        "create": [(None, None, B)],
        "p1": [([(w0, p0, u0)], None, B)],
        "p20": [(prof20, scatter, B)],
        "p4096": [(prof4096, np.arange(B), B)],
        "p20_mixed": [(mixed, scatter, B)],
        "one_handle64": [(prof64, np.repeat(np.arange(64), B // 64), B)],
        "handles64": [([pr], None, B // 64) for pr in prof64],
    }


class Arm:
    def __init__(self, torch, name, handles, dev, stream):
        self.name, self.torch = name, torch
        self.gs, self.bufs = [], []
        for profiles, cp, n in handles:
            if profiles is None:
                w, p, u = _headline()
                g = sched.Scheduler(9, w, p, u, n, device=dev.index)
            else:
                g = sched.Scheduler.from_profiles(9, profiles, cp, n_cells=n, device=dev.index)
            g.set_stream(stream.cuda_stream)
            d_cqi = torch.empty((TT, n, U, G), dtype=torch.uint8, device=dev)
            d_r2 = torch.empty((TT, n, 2), dtype=torch.int32, device=dev)
            g.synth_cqi(SEED, 0, 0, TT, d_cqi.data_ptr())
            g.synth_rand2(SEED, 0, 0, TT, d_r2.data_ptr())
            out = {"rbg_to_ue": torch.empty((TT, n, G), dtype=torch.int16, device=dev),
                   "tbs_bits": torch.empty((TT, n, U), dtype=torch.int32, device=dev),
                   "mcs": torch.empty((TT, n, U), dtype=torch.uint8, device=dev)}
            self.gs.append(g)
            self.bufs.append((n, d_cqi, d_r2, out, {k: v.data_ptr() for k, v in out.items()}))
        g0 = self.gs[0]
        self.info = {"handles": len(self.gs), "profiles": g0.n_profiles,
                     "fixed_shape": int(sched.lib().rs_fixed_shape(g0._h)),
                     "smem_bytes": g0.smem_bytes, "cells": sum(b[0] for b in self.bufs)}

    def step(self, dts):
        for g, (n, d_cqi, d_r2, _, ptrs) in zip(self.gs, self.bufs):
            g.run_device(TT, d_cqi.data_ptr(), n * U * G, d_r2.data_ptr(), dts, ptrs, ttis_per_launch=TPL)

    def close(self):
        for g in self.gs:
            g.close()


def time_arm(torch, arm, stream, dev, steps, warmup):
    _, dts = workload.tti_clock(TT)
    for _ in range(warmup):
        arm.step(dts)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    e0.record(stream)
    for _ in range(steps):
        arm.step(dts)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - wall0) * 1e3
    ms = e0.elapsed_time(e1)
    if not (0.8 * wall_ms <= ms <= 1.02 * wall_ms + 0.5):
        raise RuntimeError(f"{arm.name}: events {ms:.3f} ms disagree with the host clock {wall_ms:.3f} ms")
    return ms, wall_ms


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3, help="warm-up steps of 96 TTIs (>= 3: >= 224 TTIs)")
    ap.add_argument("--arms", default="create,p1,p20,p4096,p20_mixed,one_handle64,handles64")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("profile_bench: needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    props = torch.cuda.get_device_properties(dev)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    names = args.arms.split(",")
    table = arms(np.random.default_rng(7))
    built = {n: Arm(torch, n, table[n], dev, stream) for n in names}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in range(args.rounds):
            for n in names:
                ms, wall = time_arm(torch, built[n], stream, dev, args.steps, args.warmup)
                line = {"arm": n, "round": r, **built[n].info, "ttis_per_step": TT, "ttis_per_launch": TPL,
                        "steps": args.steps, "warmup_ttis": args.warmup * TT, "ms": round(ms, 3), "wall_ms": round(wall, 3),
                        "cell_ttis_per_s": B * TT * args.steps / (ms * 1e-3), "gpu": props.name, "power_limit": power}
                f.write(json.dumps(line) + "\n")
                f.flush()
                print(json.dumps(line), flush=True)
    for a in built.values():
        a.close()


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""bench.py -- scheduled cell-TTIs/s of the per-TTI downlink RBG allocation on B200.

Workload (BASELINE.json configs[1], SURVEY.md section 8(d)): a batch of 4096 independent cells per
GPU, 20 slices x 5 backlogged UEs, 100 MHz = 512 RBs = 64 RBGs, synthetic subband CQI drawn from
the cqi-traces-noise0 histogram and refreshed every TTI, RadioSaber inter-slice scheduler (id 9)
with PF enterprise schedulers.  A "step" is `--ttis-per-step` consecutive TTIs of the whole batch.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # the CUDA path (this repo)
  python bench.py --impl reference [...]                          # the reference's own CPU scheduler

One JSON line on stdout (rank 0).  `value` = cell-TTIs/s with inputs resident in HBM, timed with
CUDA events on the launching stream; `e2e` = the same metric through the host-buffer C-ABI calls
(rs_run_host_async / rs_wait, pinned host buffers) with the host<->device copies inside the timed
region, CQI reported every 40 TTIs like the reference's CQI_INTERVAL (enb-mac-entity.cc:38), and the
every-TTI CQI stream as the stated worst case next to a measured host-to-device ceiling; `roofline` =
algorithmic bytes of the TTI kernel / its launch time against the measured HBM peak; `parity_spot` =
three cells of the TIMED run replayed through the CPU oracle over every TTI of the run; `cpu_baseline`
= the CPU oracle port on this box's host cores (a reported baseline, not the target).

  --cells-total N   BASELINE configs[4]: N cells in total, block-partitioned over the ranks (strong
                    sharding: 65536 cells -> 8192 per GPU at 8 GPUs) instead of --cells per GPU.
  --dump-outputs D  after the timed steps, write what the last timed step returned (rbg_to_ue, tbs_bits, mcs of
                    rank 0's cells, [TTI][cell][...]) as D/<name>.npy: a fixed, seeded sample of cells within 64 MB.
                    Inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from radiosaber_b200 import workload  # noqa: E402

S, UES_PER_SLICE, G, R = 20, 5, 64, 512
U = S * UES_PER_SLICE
METRIC = "scheduled cell-TTIs/sec (20 slices x 5 UEs, 100 MHz)"
UNIT = "cell-TTIs/s"
SEED = 1


def slice_setup():
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))   # PF: epsilon 1, psi 1
    u2s = np.repeat(np.arange(S), UES_PER_SLICE).astype(np.int32)
    return w, p, u2s


def workload_config(args, n_gpus):
    total = args.cells_total if args.cells_total > 0 else args.cells * n_gpus
    per = f"{total} cells in total sharded over {n_gpus} GPU(s) (BASELINE configs[4])" if args.cells_total > 0 \
        else f"{args.cells} cells/GPU (BASELINE configs[1])"
    return {
        "workload": f"{per} x {S} slices x {UES_PER_SLICE} backlogged UEs, 100 MHz "
                    f"({R} RBs, {G} RBGs), RadioSaber id {args.algo}, PF enterprise schedulers, synthetic CQI "
                    f"from the cqi-traces-noise0 histogram refreshed every TTI",
        "cells_per_gpu": (total + n_gpus - 1) // n_gpus if args.cells_total > 0 else args.cells,
        "cells_total": total, "slices": S, "ues": U, "rbgs": G,
        "scheduler_id": args.algo, "ttis_per_step": args.ttis_per_step, "ttis_per_launch": args.ttis_per_launch,
        "cqi_refresh_ttis": 1, "seed": SEED,
        "l2": f"each step streams {args.cells * U * G * args.ttis_per_step / 1e6:.0f} MB of CQI per GPU "
              "(> 126 MB L2), so no input is L2-resident between timed iterations",
        "parallelism": f"cells sharded over {n_gpus} GPU(s), no data-path collective; one NCCL reduce of "
                       "per-slice stats after the timed region (rs_reduce_stats, C ABI)",
    }


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (nvidia-smi's clocks line via NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


TRAFFIC_CAPTURES = ("r02_tti_kernel_ncu_full_half_batch.csv",)


def ncu_traffic_bytes():
    """(DRAM bytes of one TTI-kernel launch, file) from the newest committed ncu --set full capture
    (dram__bytes_read.sum + dram__bytes_write.sum of a 2048-cell x 16-TTI half-batch launch).  A citation of a capture, not
    a property of this run: the file is named in the line so that a stale one is visible."""
    for fn in TRAFFIC_CAPTURES:
        try:
            tot = 0.0
            for line in open(os.path.join(ROOT, "profiles", fn)):
                name, unit, val = line.strip().split(",")[:3]
                if name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(val) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[unit]
            if tot:
                return tot, "profiles/" + fn
        except Exception:
            continue
    return None, None


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
def cpu_baseline_port(args, budget_s=12.0):
    """The CPU oracle port (oracle/rs_oracle.cpp) on every host core, on a bounded sample of the
    same workload.  Test infrastructure used as the checker-side baseline only."""
    from oracle.pyoracle import OracleScheduler
    w, p, u2s = slice_setup()
    cores = os.cpu_count() or 1
    B = min(args.cells, 64 * cores)
    o = OracleScheduler(args.algo, w, p, u2s, B, n_threads=cores)
    _, dts = workload.tti_clock(64)
    cqi = workload.synth_cqi(SEED, 0, B, 0, 2, U, G)
    r2 = workload.synth_rand2(SEED, 0, B, 0, 2, S)
    o.step(cqi[0], r2[0], dt=float(dts[0]))          # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        o.step(cqi[n & 1], r2[n & 1], dt=float(dts[1 + (n % 60)]))
        n += 1
        el = time.perf_counter() - t0
        if el > budget_s or n >= 400:
            break
    return {"value": B * n / el, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{B} cells x {n} TTIs of the same workload, oracle/rs_oracle.cpp -O2, {cores} threads, {el:.1f} s"}


def run_reference_arm(args, n_gpus):
    """`--impl reference`: the UNMODIFIED reference scheduler (DownlinkTransportScheduler::DoSchedule,
    compiled from the reference sources into oracle/_ref/ref_harness with its own -O0 flags) on the
    host cores: one single-threaded simulator process per core, one cell each, same slice config,
    same synthetic CQI / rand() streams.  Falls back to the oracle port if the harness binary is
    absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    harness = os.path.join(ROOT, "oracle", "_ref", "O2" if args.ref_opt == "O2" else "", "ref_harness")
    cfg = workload_config(args, n_gpus)
    K, W = args.steps, args.warmup
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": cfg, "gpu_launches": 0}
    if os.path.exists(harness):
        ttis_step = args.ref_ttis_per_step
        T = (K + W) * ttis_step
        procs = min(cores, args.ref_procs) if args.ref_procs > 0 else cores
        with tempfile.TemporaryDirectory() as tmp:
            json.dump({"slices": [{"n_slices": S, "weight": 1.0 / S, "video_app": 0, "video_bitrate": 0,
                                   "internet_flow": 0, "if_bitrate": 0, "backlog_flow": 1, "algo_alpha": 0,
                                   "algo_beta": 0, "algo_epsilon": 1, "algo_psi": 1}],
                       "ues_per_slice": [UES_PER_SLICE] * S}, open(os.path.join(tmp, "cfg.json"), "w"))
            running = []
            for pi in range(procs):
                workload.synth_cqi(SEED, pi, 1, 0, T, U, G)[:, 0].tofile(os.path.join(tmp, f"cqi{pi}.bin"))
                workload.synth_rand2(SEED, pi, 1, 0, T, S)[:, 0].tofile(os.path.join(tmp, f"rand{pi}.bin"))
                running.append(subprocess.Popen(
                    [harness, "--algo", str(args.algo), "--config", os.path.join(tmp, "cfg.json"),
                     "--ttis", str(T), "--cqi", os.path.join(tmp, f"cqi{pi}.bin"),
                     "--rand", os.path.join(tmp, f"rand{pi}.bin"), "--time-every", str(ttis_step)],
                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=tmp))
            cum, cum_stop = [], []
            for pr in running:
                out, _ = pr.communicate()
                marks = [json.loads(l) for l in out.splitlines() if l.startswith('{"sched_calls"')]
                cum.append([m["sched_seconds"] for m in marks][: K + W])
                cum_stop.append([m.get("stop_seconds", 0.0) for m in marks][: K + W])
        keep = [i for i, c in enumerate(cum) if len(c) == K + W]
        cum_all = np.array([cum[i] for i in keep])
        cum_alloc = cum_all - np.array([cum_stop[i] for i in keep]) if keep else cum_all
        cum = cum_alloc if args.ref_region == "alloc" else cum_all
        if cum.size == 0:
            print(json.dumps({"impl": "reference", "unavailable": "ref_harness produced no timing"}))
            return
        # per step: the slowest process defines the step time (all processes run concurrently)
        steps = np.diff(np.concatenate([np.zeros((cum.shape[0], 1)), cum], axis=1), axis=1)[:, W:]
        step_s = steps.max(axis=0)
        total = float(step_s.sum())
        value = cum.shape[0] * ttis_step * K / total
        region = ("EWMA + SelectFlowsToSchedule + RBsAllocation (DoSchedule minus DoStopSchedule: no RLC, packets or cerr lines)"
                  if args.ref_region == "alloc" else
                  "the reference's DoSchedule (EWMA + SelectFlows + RBsAllocation + DoStopSchedule)")
        kind, sample = "reference", (f"{cum.shape[0]} single-threaded LTE-Sim processes (one per core) x {ttis_step} TTIs "
                                     f"per step, 1 cell each; timed region = {region}, "
                                     f"-{args.ref_opt}{' as shipped' if args.ref_opt == 'O0' else ' (second build, oracle/_ref/O2)'}")
        ms = 1e3 * total / K
        ncores = int(cum.shape[0])

        def rate(c):   # cell-TTIs/s summed over the processes, timed steps only
            st = np.diff(np.concatenate([np.zeros((c.shape[0], 1)), c], axis=1), axis=1)[:, W:]
            return float(c.shape[0] * ttis_step * K / st.max(axis=0).sum())
        line["reference_regions"] = {
            "build": "-" + args.ref_opt, "cores": ncores,
            "do_schedule": {"summed": rate(cum_all), "per_core": rate(cum_all) / ncores},
            "ewma_select_alloc": {"summed": rate(cum_alloc), "per_core": rate(cum_alloc) / ncores},
            "note": "SURVEY 8(d): the allocation region excludes DoStopSchedule (byte accounting interleaved with RLC / "
                    "packet objects / cerr); BASELINE.md section 3"}
    else:
        base = cpu_baseline_port(args, budget_s=20.0)
        value, kind, sample, ms, ncores = base["value"], "port", base["sample"], None, base["cores"]
    line.update({"value": value, "ms_per_step": ms,
                 "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncores, "kind": kind, "sample": sample},
                 "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def pinned(nbytes, write_combined=False):
    """uint8 numpy view of page-locked host memory from the library (rs_host_alloc)."""
    import ctypes as C
    from radiosaber_b200 import sched
    ptr = C.c_void_p()
    sched._check(sched.lib().rs_host_alloc(int(nbytes), 1 if write_combined else 0, C.byref(ptr)))
    buf = (C.c_uint8 * int(nbytes)).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=np.uint8)
    return arr, ptr


DUMP_BYTES = 60_000_000   # data of all --dump-outputs files: under 64 MB with room for the .npy headers
DUMP_TYPES = {"rbg_to_ue": np.float32, "tbs_bits": np.float64, "mcs": np.float32}   # exact for int16 / int32 / uint8


def dump_outputs(path, outs):
    """Writes the [TTI][cell][...] device arrays `outs` as path/<name>.npy.  A batch over DUMP_BYTES keeps a seeded
    choice of cells (the same on every run with the same arguments) and, for very long steps, the last TTIs."""
    import torch
    TT, B = outs["rbg_to_ue"].shape[:2]
    per_cell_tti = sum(t[0, 0].numel() * np.dtype(DUMP_TYPES[k]).itemsize for k, t in outs.items())
    n_tti = min(TT, DUMP_BYTES // per_cell_tti)
    n_cells = min(B, DUMP_BYTES // (per_cell_tti * n_tti))
    cells = np.sort(np.random.default_rng(SEED).choice(B, n_cells, replace=False))
    idx = torch.from_numpy(cells).to(outs["rbg_to_ue"].device)
    os.makedirs(path, exist_ok=True)
    for k, t in outs.items():
        np.save(os.path.join(path, k + ".npy"), t[TT - n_tti:].index_select(1, idx).cpu().numpy().astype(DUMP_TYPES[k]))


def oracle_spot_check(args, g, cells, cell0, n_ttis, period, dts, last_out, last_t0):
    """Replays `cells` of the timed device-resident run through the CPU oracle for all n_ttis TTIs (TTI n read CQI /
    rand() slab n % period) and compares the final state of those cells and the outputs of the run's last step."""
    from oracle.pyoracle import OracleScheduler
    w, p, u2s = slice_setup()
    st = g.get_state()
    o = OracleScheduler(args.algo, w, p, u2s, len(cells))
    cqi = np.stack([workload.synth_cqi(SEED, cell0 + c, 1, 0, period, U, G)[:, 0] for c in cells], axis=1)   # [period][n][U][G]
    r2 = np.stack([workload.synth_rand2(SEED, cell0 + c, 1, 0, period, S)[:, 0] for c in cells], axis=1)
    bad = 0
    for n in range(n_ttis):
        out = o.step(cqi[n % period], r2[n % period], dt=float(dts[n]))
        if n >= last_t0:
            for k in ("rbg_to_ue", "tbs_bits", "mcs"):
                bad += int(not np.array_equal(out[k], last_out[k][n - last_t0][cells]))
    so = o.get_state()
    fields = ["avg_rate", "tx_bytes", "cum_bytes", "cum_rbs"] + (["slice_offset"] if args.algo in (8, 9, 10, 101, 103) else []) \
        + (["nvs_ewma"] if args.algo in (7, 11) else [])
    for k in fields:
        bad += int(not np.array_equal(so[k], st[k][cells]))
    return {"cells": len(cells), "ttis": int(n_ttis), "mismatches": int(bad),
            "compared": f"final {'/'.join(fields)} of cells {list(map(int, cells))} after every TTI of the run (warm-up + timed) "
                        f"and rbg_to_ue/tbs_bits/mcs of the last {n_ttis - last_t0} TTIs, against oracle/rs_oracle.cpp"}


def run_cuda_arm(args, n_gpus):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from radiosaber_b200 import sched, shard

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's "NCCL version ..." banner at
    # communicator creation, for one) is sent to stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local_rank if world > 1 else 0)
    if world > 1:
        # one process per GPU: run on (and, by first touch, take pinned host memory from) the cores next to it,
        # otherwise the end-to-end legs of all ranks pull their CQI through one socket
        try:
            import pynvml
            pynvml.nvmlInit()
            words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(dev.index), (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
            if cpus:
                os.sched_setaffinity(0, cpus & os.sched_getaffinity(0) or cpus)
        except Exception:
            pass
    TT, K, W = args.ttis_per_step, args.steps, args.warmup
    if args.cells_total > 0:     # BASELINE configs[4]: a fixed batch, block-partitioned over the ranks
        cell0, B = shard.shard_cells(args.cells_total, world, rank)
        total_cells = args.cells_total
    else:                         # configs[1]: --cells per GPU, every rank its own Monte-Carlo cells
        B = args.cells
        cell0, _ = shard.shard_cells(B * world, world, rank)
        total_cells = B * world
    w, p, u2s = slice_setup()
    g = sched.Scheduler(args.algo, w, p, u2s, B, device=dev.index)
    # a stream of our own, made current: the kernels, the generators and the timing events all go to it.  (The legacy
    # default stream has handle 0, which rs_set_stream reads as "the handle's own stream": events recorded on the
    # default stream would then not be ordered after the kernels.  Round 1 timed that way and hid it behind a host
    # synchronisation per step -- the last step's kernels were outside its events.)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    g.set_stream(stream.cuda_stream)

    # inputs resident in HBM before the timed region: CQI and rand() streams of one step's TTIs
    d_cqi = torch.empty((TT, B, U, G), dtype=torch.uint8, device=dev)
    d_r2 = torch.empty((TT, B, 2), dtype=torch.int32, device=dev)
    g.synth_cqi(SEED, cell0, 0, TT, d_cqi.data_ptr())
    g.synth_rand2(SEED, cell0, 0, TT, d_r2.data_ptr())
    d_rbg = torch.empty((TT, B, G), dtype=torch.int16, device=dev)
    d_bits = torch.empty((TT, B, U), dtype=torch.int32, device=dev)
    d_mcs = torch.empty((TT, B, U), dtype=torch.uint8, device=dev)
    outs = {"rbg_to_ue": d_rbg.data_ptr(), "tbs_bits": d_bits.data_ptr(), "mcs": d_mcs.data_ptr()}
    _, dts = workload.tti_clock((W + K) * TT)

    def step(k):
        g.run_device(TT, d_cqi.data_ptr(), B * U * G, d_r2.data_ptr(), dts[k * TT:(k + 1) * TT], outs,
                     ttis_per_launch=args.ttis_per_launch)

    for k in range(W):
        step(k)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(dev.index)
    sampler.start()
    launches0 = g.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    wall0 = time.perf_counter()
    e0.record(stream)
    for k in range(W, W + K):
        step(k)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - wall0) * 1e3
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    sampler.join()
    ms = e0.elapsed_time(e1)
    # the device clock and the host clock around the same synchronised region must tell the same story
    if not (0.8 * wall_ms <= ms <= 1.02 * wall_ms + 0.5):
        raise RuntimeError(f"timing events ({ms:.3f} ms) disagree with the host clock ({wall_ms:.3f} ms): the kernels are "
                           "not on the stream the events were recorded on")
    launches = g.launch_count - launches0
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    tl = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tl, op=dist.ReduceOp.SUM)
    ms_max = float(tms.item())
    value = total_cells * TT * K / (ms_max * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rbg_to_ue": d_rbg, "tbs_bits": d_bits, "mcs": d_mcs})

    # ---- the run that was just timed, checked: three of its cells through the CPU oracle, every TTI ----------
    parity_spot = None
    if rank == 0 and not args.no_parity_spot:
        last = {"rbg_to_ue": d_rbg.cpu().numpy(), "tbs_bits": d_bits.cpu().numpy(), "mcs": d_mcs.cpu().numpy()}
        cells = sorted({0, B // 2, B - 1})
        parity_spot = oracle_spot_check(args, g, np.array(cells), cell0, (W + K) * TT, TT, dts, last, (W + K - 1) * TT)

    # ---- end-of-run per-slice totals: the single NCCL reduce of the north star, from C (rs_reduce_stats) -------
    stats_how = "rs_get_stats (one GPU: nothing to reduce)"
    stats = g.get_stats()
    if world > 1:
        try:
            Ln = C.CDLL(os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so"))
            Ln.rs_nccl_last_error.restype = C.c_char_p
            uid = torch.zeros(128, dtype=torch.uint8)
            if rank == 0:
                raw = (C.c_uint8 * 128)()
                assert Ln.rs_comm_unique_id(raw) == 0, Ln.rs_nccl_last_error()
                uid = torch.tensor(list(raw), dtype=torch.uint8)
            uid = uid.to(dev)
            dist.broadcast(uid, src=0)      # the id travels through the launcher's process group
            raw = (C.c_uint8 * 128)(*uid.cpu().tolist())
            comm = C.c_void_p()
            assert Ln.rs_comm_init_rank(world, rank, raw, dev.index, C.byref(comm)) == 0, Ln.rs_nccl_last_error()
            red = np.zeros((4, S), dtype=np.uint64)
            Ln.rs_reduce_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
            assert Ln.rs_reduce_stats(g._h, comm, 0, red.ctypes.data_as(C.c_void_p)) == 0, Ln.rs_nccl_last_error()
            Ln.rs_comm_destroy.argtypes = [C.c_void_p]
            Ln.rs_comm_destroy(comm)
            stats = red
            stats_how = "rs_reduce_stats (include/rs_sched_nccl.h): ncclReduce(sum, root 0) of uint64 [4][S] on the handle's stream"
        except Exception as exc:   # the statistic is not the measurement: fall back to the launcher's collective, and say so
            d_stats = torch.from_numpy(stats.view(np.int64).copy()).to(dev)
            shard.reduce_stats(d_stats, dst=0)
            stats = d_stats.cpu().numpy().view(np.uint64)
            stats_how = f"torch.distributed.reduce (rs_reduce_stats unavailable: {exc})"

    # ---- end to end through the host-buffer C-ABI calls (pinned host memory, copies timed) ---------------
    # A step = TE TTIs through rs_run_host_async; the loop alternates two sets of result buffers and reads step k-1's
    # results on the host (rs_wait) while step k is in flight, so the slot ring never drains between calls.
    # Headline: CQI in the 4-bit wire layout reported every 40 TTIs (the reference's CQI_INTERVAL).  Variants: fresh
    # CQI every TTI (worst case: PCIe- / host-memory-bound, shown against a measured copy ceiling), the u8 layout, and
    # trace replay.
    TE = args.e2e_ttis
    KE = max(2, min(K, args.e2e_steps))
    # one continuing TTI clock over all calls (warm-up included), like the device-resident leg: restarting it would
    # hand every call a first TTI with dt = 7e-17 s and a non-zero byte count, i.e. a burst in the EWMA rates
    now_e, dte_all = workload.tti_clock((2 + KE) * TE)
    lib = sched.lib()

    def host_results():
        rbg, p1 = pinned(TE * B * G * 2)
        bits, p2 = pinned(TE * B * U * 4)
        mcs, p3 = pinned(TE * B * U)
        o = sched._Out(p1, p2, p3, None, None, None, None, None, None, None)
        return {"rbg": rbg.view(np.int16), "bits": bits.view(np.int32), "mcs": mcs, "o": o, "ptrs": (p1, p2, p3)}

    def timed_async_loop(call):
        """call(k, results) -> ticket.  Two warm-up steps, then KE timed steps; returns (seconds, checksum)."""
        res = [host_results(), host_results()]
        tickets = {}
        for k in range(2):
            tickets[k] = call(k, res[k & 1])
        sched._check(lib.rs_sync(ge_box[0]._h))
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        acc = 0
        t0 = time.perf_counter()
        for k in range(2, 2 + KE):
            tickets[k] = call(k, res[k & 1])
            if k > 2:
                sched._check(lib.rs_wait(ge_box[0]._h, tickets[k - 1]))
                acc += int(res[(k - 1) & 1]["bits"][-1])          # the step's results are read on the host
        sched._check(lib.rs_wait(ge_box[0]._h, tickets[1 + KE]))
        acc += int(res[(1 + KE) & 1]["bits"][-1])
        el = time.perf_counter() - t0
        te = torch.tensor([el], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        sched._check(lib.rs_sync(ge_box[0]._h))
        for r in res:
            for ptr in r["ptrs"]:
                lib.rs_host_free(ptr)
        return float(te.item()), acc

    ge_box = [None]

    def e2e_run(layout, refresh, tpl):
        ge = sched.Scheduler(args.algo, w, p, u2s, B, device=dev.index, cqi_per_rb=layout)
        ge_box[0] = ge
        n_slabs = -(-TE // refresh)
        row = G // 2 if layout == 2 else G
        d_tmp = torch.empty((n_slabs, B, U, row), dtype=torch.uint8, device=dev)
        ge.synth_cqi(SEED, cell0, 0, n_slabs, d_tmp.data_ptr())
        ge.sync()
        h_cqi, p_cqi = pinned(n_slabs * B * U * row, write_combined=args.e2e_write_combined)
        torch.from_numpy(h_cqi).copy_(d_tmp.reshape(-1))
        del d_tmp
        h_r2, p_r2 = pinned(TE * B * 2 * 4, write_combined=args.e2e_write_combined)
        h_r2.view(np.int32)[:] = workload.synth_rand2(SEED, cell0, B, 0, TE, S).reshape(-1)

        def call(k, r):
            dte = dte_all[k * TE:(k + 1) * TE]
            tk = C.c_int64(-1)
            sched._check(lib.rs_run_host_async(ge._h, TE, p_cqi, refresh, p_r2, None, dte.ctypes.data_as(C.c_void_p),
                                               C.byref(r["o"]), tpl, C.byref(tk)))
            return int(tk.value)

        el, _ = timed_async_loop(call)
        ge.close()
        lib.rs_host_free(p_cqi)
        lib.rs_host_free(p_r2)
        h2d = n_slabs * B * U * row + TE * (B * 2 * 4)
        d2h = TE * (B * G * 2 + B * U * 4 + B * U)
        return total_cells * TE * KE / el, h2d, d2h

    def e2e_trace_run():
        """Trace-driven variant (SURVEY 8 a16): 158 synthetic traces x 475 lines of the same CQI histogram
        resident in HBM (4-bit, 2.4 MB), every (cell, UE) replays a random one, a report every 40 TTIs as in
        the reference; only rand2 goes up, the same results come down."""
        ge = sched.Scheduler(args.algo, w, p, u2s, B, device=dev.index, cqi_per_rb=2)
        ge_box[0] = ge
        rng = np.random.default_rng(SEED + rank)
        traces = np.repeat(workload.histogram_cqi(rng, (158, 475, G)), 8, axis=2)
        ge.set_traces(traces, rng.integers(0, 158, (B, U)).astype(np.int32))
        rows_all = sched.trace_rows_for_run(now_e, 0)
        h_r2, p_r2 = pinned(TE * B * 2 * 4)
        h_r2.view(np.int32)[:] = workload.synth_rand2(SEED, cell0, B, 0, TE, S).reshape(-1)

        def call(k, r):
            rows, dte = rows_all[k * TE:(k + 1) * TE], dte_all[k * TE:(k + 1) * TE]
            tk = C.c_int64(-1)
            sched._check(lib.rs_run_traces_host_async(ge._h, TE, rows.ctypes.data_as(C.c_void_p), p_r2, None,
                                                      dte.ctypes.data_as(C.c_void_p), C.byref(r["o"]),
                                                      args.e2e_trace_ttis_per_launch, C.byref(tk)))
            return int(tk.value)

        el, _ = timed_async_loop(call)
        ge.close()
        lib.rs_host_free(p_r2)
        return total_cells * TE * KE / el, TE * (B * 2 * 4)

    def h2d_ceiling(nbytes_per_copy, copies):
        """What this host gives this rank when every rank copies at once and nothing else runs: `copies` pinned
        host-to-device copies of the streaming leg's chunk size, GB/s per rank (max time over ranks)."""
        src, p_src = pinned(nbytes_per_copy, write_combined=args.e2e_write_combined)
        src[:] = 7
        dst = torch.empty(nbytes_per_copy, dtype=torch.uint8, device=dev)
        hsrc = torch.from_numpy(src)
        cs = torch.cuda.Stream(dev)
        with torch.cuda.stream(cs):
            dst.copy_(hsrc, non_blocking=True)
        cs.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(cs):
            for _ in range(copies):
                dst.copy_(hsrc, non_blocking=True)
        cs.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        lib.rs_host_free(p_src)
        return nbytes_per_copy * copies / float(te.item()) / 1e9

    if args.kernel_only:   # development aid: the device-resident number alone (not a valid bench line)
        if rank == 0:
            emit({"kernel_only": True, "value": value, "ms_per_step": ms_max / K,
                  "smem_bytes_per_cta": g.smem_bytes, "clocks": sampler.result(), "parity_spot": parity_spot})
        g.close()
        if world > 1:
            dist.destroy_process_group()
        return
    e2e_value, h2d, d2h = e2e_run(2, 40, args.e2e_refresh_ttis_per_launch)
    e2e_r1, h2d_r1, _ = e2e_run(2, 1, args.e2e_ttis_per_launch)
    e2e_u8, h2d_u8, _ = e2e_run(0, 1, args.e2e_ttis_per_launch)
    e2e_tr, h2d_tr = e2e_trace_run()
    chunk_bytes = args.e2e_ttis_per_launch * B * U * (G // 2)
    ceil_gbs = h2d_ceiling(chunk_bytes, max(4, (TE * KE) // args.e2e_ttis_per_launch))
    r1_gbs = e2e_r1 / world * (h2d_r1 / (B * TE)) / 1e9           # bytes/s this rank's every-TTI leg pulled up

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        alg = g.algorithmic_bytes_per_cell_tti
        # a big batch runs as two half-batch launches per chunk of TTIs, chained on two streams so that they overlap
        # (DESIGN.md): the launch duration that the timed region supports is the region divided by the launches in it
        launches_rank0 = launches
        chunks = K * ((TT + args.ttis_per_launch - 1) // args.ttis_per_launch)
        halves = max(1, launches_rank0 // chunks)
        launch_ms = ms_max / launches_rank0
        ttis_launch = min(TT, args.ttis_per_launch)
        cells_launch = B / halves
        achieved = alg * cells_launch * ttis_launch / (launch_ms * 1e-3) / 1e9
        traffic, traffic_file = ncu_traffic_bytes()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "wall_ms_per_step_rank0": wall_ms / K, "higher_is_better": True,
            "scaling": "strong" if args.cells_total > 0 else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
            "gpu_launches": int(tl.item()),
            "parity_spot": parity_spot,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ttis_per_step": TE, "steps": KE,
                    "api": "rs_run_host_async + rs_wait (C ABI, page-locked host buffers from rs_host_alloc, copies "
                           "overlapped with kernels, two alternating result sets read on the host every step); CQI in "
                           "the 4-bit layout (cqi_per_rb=2) reported every 40 TTIs = the reference's CQI_INTERVAL "
                           "(enb-mac-entity.cc:38)",
                    "variants": {"packed_cqi_every_tti": {
                                     "value": e2e_r1, "h2d_bytes_per_step": h2d_r1,
                                     "note": "worst case: 3200 B of fresh CQI per cell-TTI; bound by the host-to-device "
                                             "path, not by the kernel",
                                     "h2d_gbs_per_gpu": r1_gbs, "h2d_ceiling_gbs_per_gpu": ceil_gbs,
                                     "frac_of_h2d_ceiling": r1_gbs / ceil_gbs if ceil_gbs else None,
                                     "ceiling": f"{world} rank(s) copying {chunk_bytes} B chunks from pinned memory at once, "
                                                "no kernels, max time over ranks"},
                                 "u8_cqi_every_tti": {"value": e2e_u8, "h2d_bytes_per_step": h2d_u8},
                                 "trace_replay_refresh40": {"value": e2e_tr, "h2d_bytes_per_step": h2d_tr,
                                                            "api": "rs_run_traces_host_async: CQI replayed from 158 traces resident in HBM"}}},
            "roofline": {"bound": "hbm", "kernel": f"rs_tti_kernel<{args.algo}>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic if (cells_launch, ttis_launch) == (2048, 16) else None,
                         "traffic_note": f"DRAM bytes of one launch (2048 cells x 16 TTIs), ncu --set full, {traffic_file} "
                                         "(a committed capture, not measured by this run)",
                         "algorithmic_bytes_per_launch": alg * cells_launch * ttis_launch, "peak_source": peak_src,
                         "algorithmic_bytes_per_cell_tti": alg, "cell_ttis_per_launch": cells_launch * ttis_launch,
                         "launch_ms": launch_ms, "launches_in_timed_region": int(launches_rank0),
                         "launch_note": f"{halves} half-batch launch(es) per {ttis_launch}-TTI chunk, overlapping on two streams: "
                                        "launch_ms = timed region / launches in it",
                         "note": "path is bound by shared-memory sort/scan and FP64 issue, not HBM (DESIGN.md)"},
            "clocks": sampler.result(),
            "smem_bytes_per_cta": g.smem_bytes,
            "kernel_instantiation": ("FixedShape<20,5,64,8,%d>" % (0 if sched.lib().rs_fixed_shape(g._h) == 0 else 2))
            if sched.lib().rs_fixed_shape(g._h) >= 0 else "DynShape (general kernel)",
            "stats_reduce": stats_how,
            "slice_bytes_total": [int(x) for x in stats[0]],
            "jain_fairness_per_slice_mean": float(np.mean(sched.jain_index(stats, np.full(S, UES_PER_SLICE * total_cells)))),
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_port(args)
        emit(line)
    g.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--cells", type=int, default=4096, help="cells per GPU")
    ap.add_argument("--algo", type=int, default=9)
    ap.add_argument("--ttis-per-step", type=int, default=96)
    ap.add_argument("--ttis-per-launch", type=int, default=16)
    ap.add_argument("--e2e-ttis", type=int, default=80)
    ap.add_argument("--e2e-ttis-per-launch", type=int, default=8)
    ap.add_argument("--e2e-write-combined", action="store_true", help="write-combined pinned input buffers")
    ap.add_argument("--cells-total", type=int, default=0, help="BASELINE configs[4]: total cells, sharded over the ranks")
    ap.add_argument("--no-parity-spot", action="store_true")
    ap.add_argument("--e2e-trace-ttis-per-launch", type=int, default=16)
    ap.add_argument("--e2e-refresh-ttis-per-launch", type=int, default=10, help="headline e2e leg (a CQI slab every 40 TTIs)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--ref-ttis-per-step", type=int, default=10)
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-opt", default="O0", choices=["O0", "O2"], help="reference build: -O0 as shipped, or oracle/_ref/O2")
    ap.add_argument("--ref-region", default="all", choices=["all", "alloc"],
                    help="timed region of the reference arm: all of DoSchedule, or without DoStopSchedule")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernel-only", action="store_true", help="development: skip the e2e and CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results (a seeded sample of rank 0's cells) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs needs --impl cuda")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: launch ourselves the way the driver does
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                  f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                  "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:])
    n_gpus = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    if args.impl == "reference":
        run_reference_arm(args, n_gpus)
    else:
        run_cuda_arm(args, n_gpus)


if __name__ == "__main__":
    main()

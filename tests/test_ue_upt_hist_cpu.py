"""CPU: workload.ue_upt_hist, the twin of the device's throughput-over-active-time histograms (rs_enable_ue_upt_hist),
against a plain per-UE statement of the rule; the NULL-handle refusals of the new entry points; the arguments
rs_batch --upt-bin-bytes refuses before a handle exists; and the NCCL header's export."""
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
M64 = 1 << 64
BACKLOGGED = 100000000


def loop_hist(queue, start, end, u2s, S, n_bins, bin_bytes, cell_profile):
    """The rule as include/rs_sched.h states it, one UE at a time, in Python integers."""
    T, B, U = queue.shape[:3]
    out = np.zeros((u2s.shape[0], S, n_bins), np.uint64)
    for b in range(B):
        p = int(cell_profile[b])
        for u in range(U):
            k = sum(1 for t in range(T) if any(int(x) > 0 for x in np.atleast_1d(queue[t, b, u])))
            if k == 0:
                continue
            c0 = sum(int(x) for x in np.atleast_1d(start[b, u])) % M64
            c1 = sum(int(x) for x in np.atleast_1d(end[b, u])) % M64
            d = (c1 - c0) % M64
            out[p, int(u2s[p, u]), min(d // k // bin_bytes, n_bins - 1)] += np.uint64(1)
    return out


def _case(seed, nb, P, n_bins, bin_bytes, T=13, B=7, U=9, S=4, base=0, spread=60000):
    """Queues with idle UEs (never active), a backlogged slot next to a FIFO slot (two bearers), and byte counters."""
    rng = np.random.default_rng(seed)
    shape = (B, U) if nb == 1 else (B, U, 2)
    q = np.where(rng.random((T,) + shape) < 0.6, 0, rng.integers(1, 20000, (T,) + shape)).astype(np.int32)
    q[:, :, 0] = 0                                      # UE 0 of every cell never has data: no sample
    q[:, :, 1] = np.where(np.arange(T) == 3, 40, 0).reshape((T, 1) + (1,) * (nb - 1))   # one active TTI
    if nb == 2:
        q[:, :, 2, 0] = BACKLOGGED                      # a backlogged slot next to a FIFO slot: active every TTI
    else:
        q[:, :, 2] = BACKLOGGED
    start = (np.uint64(base) + rng.integers(0, 1 << 20, shape).astype(np.uint64)).astype(np.uint64)
    add = rng.integers(0, spread, shape).astype(np.uint64) * (rng.random(shape) < 0.8)
    with np.errstate(over="ignore"):
        end = start + add.astype(np.uint64)
    u2s = np.stack([rng.integers(0, S, U) for _ in range(P)])
    cp = rng.integers(0, P, B)
    want = loop_hist(q, start, end, u2s, S, n_bins, bin_bytes, cp)
    got = workload.ue_upt_hist(q, start, end, u2s if P > 1 else u2s[0], S, n_bins, bin_bytes, cp if P > 1 else None)
    return got, want


@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("P", [1, 3])
def test_twin_equals_ue_loop(nb, P):
    got, want = _case(10 * nb + P, nb, P, 30, 300)
    assert got.dtype == np.uint64 and got.shape == want.shape
    assert np.array_equal(got, want)
    assert want[..., 0].sum() > 0 and want[..., 1:-1].sum() > 0
    assert want.sum() <= 7 * 8                          # UE 0 of each cell adds nothing


def test_one_bin_unit_bins_and_overflow():
    got, want = _case(1, 2, 3, 1, 300)
    assert np.array_equal(got, want) and want[..., 0].sum() == want.sum() > 0   # n_bins = 1: every sample in bin 0
    got, want = _case(2, 1, 1, 1 << 16, 1, spread=50000)
    assert np.array_equal(got, want) and np.count_nonzero(want) > 30             # bin_bytes = 1: bin = bytes per TTI
    got, want = _case(3, 2, 1, 6, 3000)
    assert np.array_equal(got, want) and want[..., -1].sum() > 0                 # 15 000 bytes per TTI and more


def test_inactive_ue_adds_no_sample():
    """A UE that never had data queued adds nothing, whatever its counters did; one active TTI divides by one."""
    q = np.zeros((5, 1, 3), np.int32)
    q[2, 0, 1] = 7
    q[:, 0, 2] = BACKLOGGED
    start = np.zeros((1, 3), np.uint64)
    end = np.array([[5000, 900, 5000]], np.uint64)
    h = workload.ue_upt_hist(q, start, end, [0, 1, 2], 3, 2000, 1)
    assert h.sum() == 2 and h[0, 0].sum() == 0 and h[0, 1, 900] == 1 and h[0, 2, 1000] == 1


@pytest.mark.parametrize("nb", [1, 2])
def test_deltas_across_2_32_and_the_2_64_wrap(nb):
    got, want = _case(4, nb, 1, 40, 200, base=(1 << 32) - 30000)             # counters cross 2^32 in the window
    assert np.array_equal(got, want) and want[..., 1:].sum() > 0
    got, want = _case(5, nb, 3, 40, 200, base=M64 - (1 << 20) - 30000)      # ... and wrap past 2^64
    assert np.array_equal(got, want) and want[..., 1:].sum() > 0
    q = np.ones((2, 1, 2) if nb == 1 else (2, 1, 2, 2), np.int32)
    start = np.full((1, 2) if nb == 1 else (1, 2, 2), M64 - 100, np.uint64)
    end = np.array([[50, M64 - 100]] if nb == 1 else [[[50, 0], [M64 - 100, M64 - 100]]], np.uint64)
    h = workload.ue_upt_hist(q, start, end, [0, 1], 2, 400, 1)
    assert h[0, 0].argmax() == (75 if nb == 1 else 125) and h[0, 1, 0] == 1   # a wrapped counter over 2 TTIs; idle


def test_entry_points_refuse_a_null_handle():
    """The C ABI checks the handle first (no GPU needed)."""
    L = sched.lib()
    assert L.rs_enable_ue_upt_hist(None, 8, 1000) == 1
    assert L.rs_enable_ue_upt_hist(None, 0, 0) == 1
    assert L.rs_ue_upt_hist_bins(None) == 0
    assert L.rs_ue_upt_hist_device(None, None) == 1
    assert L.rs_get_ue_upt_hist(None, None) == 1
    assert b"null handle" in L.rs_last_error() or b"bad argument" in L.rs_last_error()


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "12",
                           "--config", os.path.join(ROOT, "tests", "data", "cfg20x5_ab.json"), *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_rs_batch_argument_errors():
    traffic = os.path.join(ROOT, "tests", "data", "traffic20x5_video_voip.json")
    rate = ["--rate-window", 4, "--rate-bins", 10, "--rate-bin-bytes", 100]
    needs = "rs_batch: --upt-bin-bytes needs --buffers K and --rate-window W --rate-bins N --rate-bin-bytes X\n"
    for partial in ([], rate, ["--buffers", 4, "--traffic", traffic]):
        r = _batch(*partial, "--upt-bin-bytes", 100)
        assert r.returncode == 1 and r.stderr == needs, partial
    for x in (0, -5):
        r = _batch("--buffers", 4, "--traffic", traffic, *rate, "--upt-bin-bytes", x)
        assert r.returncode == 1 and r.stderr == "rs_batch: --upt-bin-bytes X: X bytes per TTI per bin, >= 1\n"
    r = subprocess.run([BIN, "--cells", "4"], capture_output=True, text=True)
    assert r.returncode == 2 and "[--upt-bin-bytes X]" in r.stderr


def test_nccl_ue_upt_header_symbol_is_exported():
    """include/rs_sched_nccl_ue_upt.h declares one entry point of radiosaber_b200/librs_nccl.so and redeclares none of
    the other four NCCL headers' (loads without a GPU; the one call made fails on its NULL handle before any CUDA)."""
    import ctypes
    import re
    import torch  # noqa: F401  -- before the library: a process that loads the system libnccl first cannot import torch later

    def declared(name):
        src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", name)).read(), flags=re.S)
        return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", src)))

    names = declared("rs_sched_nccl_ue_upt.h")
    assert names == ["rs_reduce_ue_upt_hist"]
    others = set().union(*[declared(h) for h in ("rs_sched_nccl.h", "rs_sched_nccl_buffers.h", "rs_sched_nccl_hol_hist.h",
                                                 "rs_sched_nccl_ue_rate.h")])
    assert not set(names) & others
    L = ctypes.CDLL(os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so"))
    assert hasattr(L, "rs_reduce_ue_upt_hist")
    L.rs_reduce_ue_upt_hist.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    L.rs_nccl_last_error.restype = ctypes.c_char_p
    assert L.rs_reduce_ue_upt_hist(None, None, 0, None) != 0
    assert b"rs_reduce_ue_upt_hist" in L.rs_nccl_last_error()

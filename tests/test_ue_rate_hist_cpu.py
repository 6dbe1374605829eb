"""CPU: workload.ue_rate_hist, the twin of the device's per-UE throughput histograms (rs_enable_ue_rate_hist /
rs_close_ue_rate_window), against a plain per-UE statement of the rule; sched.hist_percentile on those histograms; the
NULL-handle refusals of the new entry points; the arguments rs_batch --rate-window refuses before a handle exists; and
the NCCL header's export."""
import math
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")
M64 = 1 << 64


def loop_hist(start, end, u2s, S, n_bins, bin_bytes, cell_profile):
    """The rule as include/rs_sched.h states it, one UE at a time, in Python integers."""
    B, U = end.shape[:2]
    out = np.zeros((u2s.shape[0], S, n_bins), np.uint64)
    for b in range(B):
        p = int(cell_profile[b])
        for u in range(U):
            c0 = sum(int(x) for x in np.atleast_1d(start[b, u])) % M64
            c1 = sum(int(x) for x in np.atleast_1d(end[b, u])) % M64
            d = (c1 - c0) % M64
            out[p, int(u2s[p, u]), min(d // bin_bytes, n_bins - 1)] += np.uint64(1)
    return out


def _counters(seed, B, U, nb, base=0, spread=60000):
    """uint64 counters at a window's start and end: base plus a few bytes, idle UEs (no bytes) among them."""
    rng = np.random.default_rng(seed)
    shape = (B, U) if nb == 1 else (B, U, 2)
    start = (np.uint64(base) + rng.integers(0, 1 << 20, shape).astype(np.uint64)).astype(np.uint64)
    add = rng.integers(0, spread, shape).astype(np.uint64) * (rng.random(shape) < 0.8)
    with np.errstate(over="ignore"):
        end = start + add.astype(np.uint64)
    return start, end


def _case(seed, nb, P, n_bins, bin_bytes, B=7, U=9, S=4, base=0, spread=60000):
    rng = np.random.default_rng(seed + 1)
    start, end = _counters(seed, B, U, nb, base, spread)
    u2s = np.stack([rng.integers(0, S, U) for _ in range(P)])
    cp = rng.integers(0, P, B)
    want = loop_hist(start, end, u2s, S, n_bins, bin_bytes, cp)
    got = workload.ue_rate_hist(start, end, u2s if P > 1 else u2s[0], S, n_bins, bin_bytes, cp if P > 1 else None)
    return got, want


@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("P", [1, 3])
def test_twin_equals_ue_loop(nb, P):
    got, want = _case(10 * nb + P, nb, P, 30, 3000)
    assert got.dtype == np.uint64 and got.shape == want.shape
    assert np.array_equal(got, want)
    assert want[..., 0].sum() > 0 and want[..., 1:-1].sum() > 0 and want.sum() == 7 * 9


def test_one_bin_unit_bins_and_overflow():
    got, want = _case(1, 2, 3, 1, 3000)
    assert np.array_equal(got, want) and want[..., 0].sum() == 7 * 9          # n_bins = 1: every UE in bin 0
    got, want = _case(2, 1, 1, 1 << 16, 1, spread=50000)
    assert np.array_equal(got, want) and np.count_nonzero(want) > 40          # bin_bytes = 1: bin = bytes
    got, want = _case(3, 2, 1, 6, 10000)
    assert np.array_equal(got, want) and want[..., -1].sum() > want[..., 0].sum()   # 50 000 bytes and more: the last bin


@pytest.mark.parametrize("nb", [1, 2])
def test_deltas_across_2_32_and_the_2_64_wrap(nb):
    got, want = _case(4, nb, 1, 40, 2000, base=(1 << 32) - 30000)             # counters cross 2^32 in the window
    assert np.array_equal(got, want) and want[..., 1:].sum() > 0
    got, want = _case(5, nb, 3, 40, 2000, base=M64 - (1 << 20) - 30000)      # ... and wrap past 2^64
    assert np.array_equal(got, want) and want[..., 1:].sum() > 0
    start = np.full((1, 2) if nb == 1 else (1, 2, 2), M64 - 100, np.uint64)
    end = np.array([[50, M64 - 100]] if nb == 1 else [[[50, 0], [M64 - 100, M64 - 100]]], np.uint64)
    h = workload.ue_rate_hist(start, end, [0, 1], 2, 400, 1)
    assert h[0, 0].argmax() == (150 if nb == 1 else 250) and h[0, 1, 0] == 1   # a wrapped counter; an idle UE: bin 0


def test_percentiles_of_twin_histograms():
    """sched.hist_percentile's rule on the twin's histograms: the sample of rank ceil(q n / 100) of the sorted bins."""
    for seed, nb, P in ((6, 1, 1), (7, 2, 3)):
        got, _ = _case(seed, nb, P, 25, 2500, B=40, U=9)
        for p, s in np.ndindex(got.shape[:2]):
            h = got[p, s]
            samples = np.repeat(np.arange(h.shape[0]), h.astype(np.int64))
            for q in (5, 50, 95):
                want = None if samples.size == 0 else int(samples[math.ceil(q * samples.size / 100) - 1])
                assert sched.hist_percentile(h, q) == want, (p, s, q)
    assert sched.hist_percentile(np.zeros(3, np.uint64), 5) is None


def test_entry_points_refuse_a_null_handle():
    """The C ABI checks the handle first (no GPU needed)."""
    L = sched.lib()
    assert L.rs_enable_ue_rate_hist(None, 8, 1000) == 1
    assert L.rs_enable_ue_rate_hist(None, 0, 0) == 1
    assert L.rs_close_ue_rate_window(None) == 1
    assert L.rs_ue_rate_hist_bins(None) == 0
    assert L.rs_ue_rate_hist_device(None, None) == 1
    assert L.rs_get_ue_rate_hist(None, None) == 1
    assert b"null handle" in L.rs_last_error() or b"bad argument" in L.rs_last_error()


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "12",
                           "--config", os.path.join(ROOT, "tests", "data", "cfg20x5_ab.json"), *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_rs_batch_argument_errors():
    together = "rs_batch: --rate-window W, --rate-bins N and --rate-bin-bytes X go together\n"
    for partial in (["--rate-window", 4], ["--rate-bins", 10], ["--rate-bin-bytes", 100],
                    ["--rate-window", 4, "--rate-bins", 10], ["--rate-bins", 10, "--rate-bin-bytes", 100],
                    ["--rate-window", 4, "--rate-bin-bytes", 100]):
        r = _batch(*partial)
        assert r.returncode == 1 and r.stderr == together, partial
    for w in (0, -3, 5, 24):
        r = _batch("--rate-window", w, "--rate-bins", 10, "--rate-bin-bytes", 100)
        assert r.returncode == 1 and r.stderr == "rs_batch: --rate-window W: W TTIs per window, >= 1 and dividing --ttis 12\n"
    for n in (0, -1, 65537):
        r = _batch("--rate-window", 4, "--rate-bins", n, "--rate-bin-bytes", 100)
        assert r.returncode == 1 and r.stderr == "rs_batch: --rate-bins N: N bins, 1..65536\n"
    for x in (0, -5):
        r = _batch("--rate-window", 4, "--rate-bins", 10, "--rate-bin-bytes", x)
        assert r.returncode == 1 and r.stderr == "rs_batch: --rate-bin-bytes X: X bytes per bin, >= 1\n"
    r = subprocess.run([BIN, "--cells", "4"], capture_output=True, text=True)
    assert r.returncode == 2 and "[--rate-window W --rate-bins N --rate-bin-bytes X]" in r.stderr


def test_nccl_ue_rate_header_symbol_is_exported():
    """include/rs_sched_nccl_ue_rate.h declares one entry point of radiosaber_b200/librs_nccl.so and redeclares none of
    the other three NCCL headers' (loads without a GPU; the one call made fails on its NULL handle before any CUDA)."""
    import ctypes
    import re
    import torch  # noqa: F401  -- before the library: a process that loads the system libnccl first cannot import torch later

    def declared(name):
        src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", name)).read(), flags=re.S)
        return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", src)))

    names = declared("rs_sched_nccl_ue_rate.h")
    assert names == ["rs_reduce_ue_rate_hist"]
    others = set().union(*[declared(h) for h in ("rs_sched_nccl.h", "rs_sched_nccl_buffers.h", "rs_sched_nccl_hol_hist.h")])
    assert not set(names) & others
    L = ctypes.CDLL(os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so"))
    assert hasattr(L, "rs_reduce_ue_rate_hist")
    L.rs_reduce_ue_rate_hist.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    L.rs_nccl_last_error.restype = ctypes.c_char_p
    assert L.rs_reduce_ue_rate_hist(None, None, 0, None) != 0
    assert b"rs_reduce_ue_rate_hist" in L.rs_nccl_last_error()

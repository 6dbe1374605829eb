"""CPU: workload.hol_hist, the twin of the device's head-of-line delay histograms (rs_enable_hol_hist), against a plain
bearer-by-bearer statement of the rule; sched.hist_percentile; and the arguments rs_batch --hol-bins refuses before a
handle exists."""
import math
import os
import subprocess

import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.helpers import ROOT

BIN = os.path.join(ROOT, "radiosaber_b200", "rs_batch")


def loop_hist(queue, hol, tbs, algo, u2s, backlogged, S, n_bins, per_unit, cell_profile):
    """The rule as include/rs_sched.h states it, one bearer at a time."""
    T, B, U = tbs.shape
    nb = queue.shape[3]
    out = np.zeros((u2s.shape[0], 2, S, n_bins), np.uint64)
    for t in range(T):
        for b in range(B):
            p = int(cell_profile[b])
            for u in range(U):
                s = int(u2s[p, u])
                avail = int(tbs[t, b, u]) // 8
                for k in range(nb - 1, -1, -1):
                    q, h = int(queue[t, b, u, k]), float(hol[t, b, u, k])
                    served = False
                    if avail > 0 and (algo == 1 or q > 0):
                        avail -= avail if algo == 1 else min(avail, q)
                        served = True
                    if backlogged[b, u, k]:
                        continue
                    d = min(math.floor(h * per_unit + 0.5), n_bins - 1)
                    if served:
                        out[p, 0, s, d] += np.uint64(1)
                    if q > 0:
                        out[p, 1, s, d] += np.uint64(1)
    return out


def _run(seed, algo, nb, P, n_bins, per_unit=1000.0, T=6, B=5, U=6, S=3):
    """Shown queues (empty, small, 100000000 for the backlogged), delays on and between 1 ms bins, tbs_bits that run
    out part-way through a UE's slots."""
    rng = np.random.default_rng(seed)
    q = rng.choice([0, 0, 40, 300, 2000, 100000000], size=(T, B, U, nb)).astype(np.int32)
    h = np.where(q > 0, rng.integers(0, 40, q.shape) * 0.001 + rng.choice([0.0, 0.0005, 0.0004999], q.shape), 0.0)
    tbs = (rng.choice([0, 8, 200, 2600, 24000], size=(T, B, U)) * rng.integers(1, 3, (T, B, U))).astype(np.int32)
    bl = rng.random((B, U, nb)) < 0.25
    q[:, bl] = 100000000
    h[:, bl] = 0.0
    u2s = np.stack([rng.integers(0, S, U) for _ in range(P)])
    cp = rng.integers(0, P, B)
    want = loop_hist(q, h, tbs, algo, u2s, bl, S, n_bins, per_unit, cp)
    got = workload.hol_hist(q if nb == 2 else q[..., 0], h if nb == 2 else h[..., 0], tbs, algo,
                            u2s if P > 1 else u2s[0], bl if nb == 2 else bl[..., 0], S, n_bins, per_unit,
                            cp if P > 1 else None)
    return got, want, q, tbs


@pytest.mark.parametrize("algo", [9, 1, 7])
@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("P", [1, 3])
def test_twin_equals_bearer_loop(algo, nb, P):
    got, want, q, tbs = _run(algo * 10 + nb + P, algo, nb, P, 30)
    assert got.dtype == np.uint64 and got.shape == want.shape
    assert np.array_equal(got, want)
    assert want[:, 0].sum() > 0 and want[:, 1].sum() > 0


def test_one_bin_and_overflow():
    got, want, q, _ = _run(5, 9, 2, 3, 1)
    assert np.array_equal(got, want) and want.sum() > 0        # n_bins = 1: every sample in the overflow bin
    got, want, _, _ = _run(6, 9, 2, 1, 8, per_unit=1000.0)
    assert np.array_equal(got, want) and want[..., -1].sum() > want[..., 0].sum()   # delays of 7 ms and more
    got, want, _, _ = _run(7, 103, 1, 1, 50, per_unit=2000.0)
    assert np.array_equal(got, want)


def test_id1_sends_without_looking_at_the_queue():
    """Id 1's stderr loop books the first slot that has a FIFO whatever it holds; the others skip an empty one."""
    q = np.array([[[[0, 0]]]], np.int32)
    h = np.array([[[[0.003, 0.0]]]])
    tbs = np.array([[[800]]], np.int32)
    bl = np.zeros((1, 1, 2), bool)
    one = workload.hol_hist(q, h, tbs, 1, [0], bl, 1, 5)
    nine = workload.hol_hist(q, h, tbs, 9, [0], bl, 1, 5)
    assert one[0, 0, 0].tolist() == [1, 0, 0, 0, 0] and not one[0, 1].any()      # slot 1 sent (hol 0), slot 0 not
    assert not nine.any()
    q[..., 1] = 50                                                               # slot 1 takes 50 of 100 bytes
    nine = workload.hol_hist(q, h, tbs, 9, [0], bl, 1, 5)
    assert nine[0, 0, 0].tolist() == [1, 0, 0, 0, 0] and nine[0, 1, 0].tolist() == [1, 0, 0, 0, 0]
    q[..., 0] = 7                                                                # ... and slot 0 the rest
    nine = workload.hol_hist(q, h, tbs, 9, [0], bl, 1, 5)
    assert nine[0, 0, 0].tolist() == [1, 0, 0, 1, 0]


def test_percentile_rule():
    assert sched.hist_percentile(np.zeros(4, np.uint64), 50) is None
    h = np.array([2, 0, 1, 1], np.uint64)   # 4 samples
    assert [sched.hist_percentile(h, q) for q in (0, 25, 50, 51, 75, 76, 99, 100)] == [0, 0, 0, 2, 2, 3, 3, 3]
    assert sched.hist_percentile([0, 0, 7], 1) == 2
    for q in (-1, 101, 50.0, True):
        with pytest.raises(ValueError):
            sched.hist_percentile(h, q)


def _batch(*args):
    assert os.path.exists(BIN), "build with make -C radiosaber_b200/csrc"
    return subprocess.run([BIN, "--algo", "9", "--cells", "4", "--ttis", "3",
                           "--config", os.path.join(ROOT, "tests", "data", "cfg20x5_ab.json"), *[str(a) for a in args]],
                          capture_output=True, text=True, timeout=120)


def test_rs_batch_argument_errors():
    traffic = os.path.join(ROOT, "tests", "data", "traffic20x5_ab.json")
    r = _batch("--hol-bins", 10)
    assert r.returncode == 1 and r.stderr == "rs_batch: --hol-bins needs --buffers K\n"
    for n in (-1, 65537):
        r = _batch("--buffers", 4, "--traffic", traffic, "--hol-bins", n)
        assert r.returncode == 1 and r.stderr == "rs_batch: --hol-bins N: N bins of one TTI, 1..65536\n"
    r = subprocess.run([BIN, "--cells", "4"], capture_output=True, text=True)
    assert r.returncode == 2 and "[--hol-bins N]" in r.stderr


def test_scheduler_refuses_without_a_handle():
    """The C ABI checks the handle first (no GPU needed)."""
    assert sched.lib().rs_enable_hol_hist(None, 8, 1000.0) == 1
    assert sched.lib().rs_hol_hist_bins(None) == 0
    assert sched.lib().rs_get_hol_hist(None, None) == 1


def test_nccl_hol_hist_header_symbol_is_exported():
    """include/rs_sched_nccl_hol_hist.h declares one entry point of radiosaber_b200/librs_nccl.so and redeclares none of
    the other two NCCL headers' (loads without a GPU; no calls made)."""
    import ctypes
    import re
    import torch  # noqa: F401  -- before the library: a process that loads the system libnccl first cannot import torch later

    def declared(name):
        src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", name)).read(), flags=re.S)
        return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", src)))

    names = declared("rs_sched_nccl_hol_hist.h")
    assert names == ["rs_reduce_hol_hist"]
    assert not set(names) & (set(declared("rs_sched_nccl.h")) | set(declared("rs_sched_nccl_buffers.h")))
    L = ctypes.CDLL(os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so"))
    assert hasattr(L, "rs_reduce_hol_hist")

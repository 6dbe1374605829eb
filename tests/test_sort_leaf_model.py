"""CPU: executable model of a leaf schedule for the std::sort emulation, checked against the real std::sort and
against the introsort emulation at forced shallow depth limits.  The device keeps the level loop down to ranges of
<= 16 and the whole-array counting sort: every device form of this schedule measured slower (profiles/README.md, r10).
This model states what such a form must compute.

The level-synchronous loop partitions ranges longer than LEAF only.  A part of <= LEAF entries is finished at once by
the warp that cut it: partitioned to the end (depth first, left part first), then stably sorted by key and written to
out[f..l).  Two facts make that exact:
  * after the introsort loop every range of <= 16 entries (or heap-sorted at the depth limit) is already ordered
    against its neighbours, so the stable sort of the whole array is the concatenation of the stable sorts of any
    ranges the loop has finished partitioning -- no whole-array pass is needed;
  * a range's result depends only on its entries and its depth, not on when it is partitioned.
The leaf decides every swap of a partition from ranks alone: with L(q) the left stoppers (key <= pivot) before q and
R(q) the right stoppers (key >= pivot) after q, a left stopper swaps iff R(q) > L(q) and a right stopper iff
L(q) > R(q); its partner is the right (left) stopper of the same rank counted from the other end.
"""
import numpy as np
import pytest

from oracle import pyoracle
from radiosaber_b200 import workload
from tests.sort_model import THRESH, _heap_sort, _median_to_first

LEAF = 128  # four entries per lane of one warp


def _eq_perm(length):
    """rs_sched.cu build_eq_table: what the recursion does to `length` equal keys."""
    a = list(range(length))
    stack = [(0, length)]
    while stack:
        f, l = stack.pop()
        while l - f > THRESH:
            m = f + (l - f) // 2
            a[f], a[m] = a[m], a[f]
            k = 0
            while f + 1 + k < l - 1 - k:
                a[f + 1 + k], a[l - 1 - k] = a[l - 1 - k], a[f + 1 + k]
                k += 1
            cut = f + 1 + (l - f - 1) // 2
            stack.append((cut, l))
            l = cut
    mid = length // 2
    return [mid if x == 0 else (0 if x == mid else x) for x in a]


def _eq_applies(key, a, f, l, levels_left, eq_max):
    p = key[a[f]]
    return (all(key[a[q]] == p for q in range(f + 1, l)) and l - f <= eq_max
            and (l - f).bit_length() <= levels_left)


def _apply_eq(a, f, l):
    seg = [a[f + t] for t in _eq_perm(l - f)]
    a[f:l] = seg


def leaf_sort(key, a, out, f, n, depth, depth_limit, eq_max):
    """One warp's leaf: a[f..f+n) is partitioned to the end and out[f..f+n) receives it stably sorted by key."""
    v = list(a[f:f + n])
    x = [None] * n      # the range's own slots of a[]: scratch once v holds the entries
    o = [None] * n      # the range's own slots of out[], written last
    s, e, d = 0, n, depth
    while True:
        if e - s > THRESH:
            if d >= depth_limit:
                _heap_sort(key, v, s, e)
            else:
                _median_to_first(key, v, s, e)
                pk = key[v[s]]
                if _eq_applies(key, v, s, e, depth_limit - d, eq_max):
                    _apply_eq(v, s, e)
                else:
                    base = s + 1
                    is_l = [key[v[q]] <= pk for q in range(base, e)]
                    is_r = [key[v[q]] >= pk for q in range(base, e)]
                    nr = sum(is_r)
                    rd = {}
                    cut = 10 ** 9
                    for i, q in enumerate(range(base, e)):
                        lq = sum(is_l[:i])             # L(q): left stoppers before q
                        rq = nr - sum(is_r[:i + 1])    # R(q): right stoppers after q
                        sl = is_l[i] and rq > lq
                        sr = is_r[i] and lq > rq
                        if sl:
                            x[base + lq] = v[q]
                            rd[q] = e - 1 - lq
                        elif sr:
                            x[e - 1 - rq] = v[q]
                            rd[q] = base + rq
                        if (is_l[i] and not sl) or sr:  # first left stopper that stays, first right one that moves
                            cut = min(cut, q)
                    for q, r in rd.items():
                        v[q] = x[r]
                    assert s < cut < e
                    x[cut], o[cut] = e, d + 1           # [cut, e) waits in its first slot
                    e, d = cut, d + 1
                    continue
        if e >= n:
            break
        s = e
        e, d = x[s], o[s]
    order = sorted(range(n), key=lambda i: -key[v[i]])   # stable
    out[f:f + n] = [v[i] for i in order]


def leaf_schedule_sort(keys, depth_limit=-1, eq_max=2048):
    """sort_desc: perm[i] = original index of the entry that ends at position i."""
    key = np.asarray(keys)
    n = len(key)
    a = list(range(n))
    out = [None] * n
    if n == 0:
        return np.array(a)
    if depth_limit < 0:
        depth_limit = 2 * (int(n).bit_length() - 1)
    eq_max = min(n, eq_max)
    if n <= LEAF:
        leaf_sort(key, a, out, 0, n, 0, depth_limit, eq_max)
        return np.array(out)
    segs = [(0, n)]
    level = 0
    while segs:
        if level >= depth_limit:
            for f, l in segs:
                _heap_sort(key, a, f, l)
                out[f:l] = a[f:l]
            break
        nxt = []
        for f, l in segs:
            _median_to_first(key, a, f, l)
            if _eq_applies(key, a, f, l, depth_limit - level, eq_max):
                _apply_eq(a, f, l)
                out[f:l] = a[f:l]
                continue
            p = key[a[f]]
            pos = np.arange(f + 1, l)
            k = key[np.asarray(a)[pos]]
            pos_l = pos[k <= p]
            pos_r = pos[k >= p][::-1]
            m = min(len(pos_l), len(pos_r))
            big_k = int((pos_l[:m] < pos_r[:m]).sum())
            cut = int(pos_l[big_k]) if big_k < len(pos_l) else 10 ** 9
            if big_k >= 1:
                cut = min(cut, int(pos_r[big_k - 1]))
            for q in range(big_k):
                a[pos_l[q]], a[pos_r[q]] = a[pos_r[q]], a[pos_l[q]]
            for pf, pl in ((f, cut), (cut, l)):
                if pl - pf <= LEAF:
                    leaf_sort(key, a, out, pf, pl - pf, level + 1, depth_limit, eq_max)
                else:
                    nxt.append((pf, pl))
        segs = nxt
        level += 1
    return np.array(out)


def _cqi_keys(rng, shape):
    p = workload.CQI_HIST.astype(np.float64) / workload.CQI_TOTAL
    return rng.choice(np.arange(1, 16), size=shape, p=p).astype(np.float64)


def _families(rng, n):
    """The key families of tests/test_gpu_parity.py::test_device_sort_matches_std_sort."""
    rows = [
        _cqi_keys(rng, n),
        rng.integers(0, 16, size=n).astype(np.float64),
        np.full(n, 7.0),
        np.sort(rng.integers(0, 16, size=n)).astype(np.float64),
        np.sort(rng.integers(0, 16, size=n))[::-1].astype(np.float64),
        np.maximum.reduce(_cqi_keys(rng, (5, n))),
        (rng.integers(0, 2, size=n) * 15).astype(np.float64),
        np.maximum.reduce(_cqi_keys(rng, (40, n))),
        rng.choice(np.array([3.0, 12.0, 13.0]), size=n, p=[0.1, 0.8, 0.1]),
    ]
    return rows


@pytest.mark.parametrize("n", [1, 2, 16, 17, 31, 32, 33, 64, 320, 448, 1280, 1290, 3200, 4096])
def test_leaf_schedule_matches_std_sort(n):
    rng = np.random.default_rng(n)
    for i, keys in enumerate(_families(rng, n)):
        assert np.array_equal(leaf_schedule_sort(keys), pyoracle.std_sort_desc(keys)), (n, i)


def test_leaf_schedule_every_length_up_to_300():
    rng = np.random.default_rng(300)
    for n in range(1, 301):
        for i, keys in enumerate(_families(rng, n)):
            assert np.array_equal(leaf_schedule_sort(keys), pyoracle.std_sort_desc(keys)), (n, i)


@pytest.mark.parametrize("depth", [0, 1, 2, 3, 4, 5, 8])
def test_leaf_schedule_depth_limit_matches_emulation(depth):
    rng = np.random.default_rng(70 + depth)
    for n in (17, 40, 100, 128, 129, 300, 1280):
        rows = _families(rng, n) + [rng.integers(0, 16, size=n).astype(np.float64) for _ in range(4)]
        for i, keys in enumerate(rows):
            want = pyoracle.introsort_emul_desc(keys, depth)
            assert np.array_equal(leaf_schedule_sort(keys, depth), want), (n, depth, i)

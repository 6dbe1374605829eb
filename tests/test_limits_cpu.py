"""UpperBound (id 10) past 2G grants, host side: the oracle's grant list at any length and the log writer fed a list
longer than 2G.  In UpperBound every slice takes its own best min(quota, G) RBGs, so a TTI can make up to S*G grants;
with many slices on few RBGs more than 2G are common (40 slices on 16 RBGs: most TTIs).  Runs without a GPU."""
import re

import numpy as np

from oracle.pyoracle import OracleScheduler, lib as oracle_lib
from radiosaber_b200 import sched, workload

# 40 slices of one or two UEs on 48 RBs in RBGs of 3 (16 RBGs): more than 2G = 32 grants from the first TTIs on
S, N_RBS, RBG, B, T = 40, 48, 3, 3, 24
G = N_RBS // RBG


def _setup(seed=3):
    rng = np.random.default_rng(seed)
    u2s = np.repeat(np.arange(S), rng.integers(1, 3, S)).astype(np.int32)
    w = rng.dirichlet(np.ones(S) * 0.5)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    return u2s, w, p


def _run(grant_list_len):
    """T TTIs of the oracle; per TTI its outputs, and the state at the end."""
    u2s, w, p = _setup()
    U = len(u2s)
    o = OracleScheduler(10, w, p, u2s, B, n_rbs=N_RBS, rbg_size=RBG, n_threads=4, grant_list_len=grant_list_len)
    _, dts = workload.tti_clock(T)
    outs = []
    for t in range(T):
        cqi = workload.synth_cqi(5, 0, B, t, 1, U, G)[0]
        outs.append(o.step(cqi, workload.synth_rand_draws(5, 0, B, t, 1, S, 2)[0], dt=float(dts[t]), want_aux=True))
    return outs, o.get_state()


def test_oracle_grant_list_is_a_prefix_at_every_length():
    """The list of length L is the first L entries of the whole list (S*G) and -1 after alloc_n; alloc_n, every other
    output and the state do not depend on L."""
    full, st_full = _run(S * G)
    n = np.stack([x["alloc_n"] for x in full])
    assert n.max() > 2 * G and (n > 2 * G).sum() > B * T // 2, n.max()
    for L in (2 * G, 2 * G + 1, 3 * G - 1, int(n.max()) - 1, int(n.max()), S * G - 7):
        part, st = _run(L)
        for t in range(T):
            for k, v in full[t].items():
                if k in ("alloc_ue", "alloc_rbg"):
                    assert np.array_equal(part[t][k], v[:, :L]), (L, t, k)
                    for b in range(B):
                        assert (v[b, n[t, b]:] == -1).all() and (v[b, :n[t, b]] >= 0).all(), (L, t, b, k)
                else:
                    assert np.array_equal(part[t][k], v), (L, t, k)
        for k in st_full:
            assert np.array_equal(st[k], st_full[k]), (L, k)


def _parse_users(text):
    """{user: [(rbg, cqi), ...]} of the "User(u) allocated RBGS: g(c) ..." lines of one TTI."""
    users = {}
    for m in re.finditer(r"^User\((\d+)\) allocated RBGS:((?: \d+\(\d+\))*) final_cqi: \d+$", text, re.M):
        users[int(m.group(1))] = [tuple(map(int, x)) for x in re.findall(r" (\d+)\((\d+)\)", m.group(2))]
    return users


def test_log_tti_grants_books_every_grant():
    """rs_log_tti_grants with the whole list of a TTI of more than 2G grants: every grant is in its user's RB list (in
    grant order) and in the all_bytes sum, and the user lines differ from the ones the first 2G grants give."""
    u2s, _, _ = _setup()
    U = len(u2s)
    full, _ = _run(S * G)
    t, b = next((t, b) for t in range(T) for b in range(B) if full[t]["alloc_n"][b] > 2 * G + G // 2)
    x = {k: v[b] for k, v in full[t].items()}
    n = int(x["alloc_n"])
    cqi = workload.synth_cqi(5, 0, B, t, 1, U, G)[0][b]
    eff = [oracle_lib().rso_efficiency_from_cqi(c) for c in range(16)]

    def log(n_grants, ue, rbg):
        lw = sched.LogWriter(10, u2s, S, n_rbs=N_RBS, rbg_size=RBG)
        lw.tti_grants(100, cqi, n_grants, ue, rbg, x["tbs_bits"], x["final_cqi"], x["slice_target"], x["slice_quota"])
        return lw.stdout, lw.stderr

    out, err = log(n, x["alloc_ue"], x["alloc_rbg"])
    want, total = {}, 0.0
    for e in range(n):
        u, g = int(x["alloc_ue"][e]), int(x["alloc_rbg"][e])
        want.setdefault(u, []).append((g, int(cqi[u, g])))
        total += eff[int(cqi[u, g])]
    assert _parse_users(out) == want
    assert sum(len(v) for v in want.values()) == n > 2 * G
    assert re.search(r"^all_bytes: (\d+)$", err, re.M).group(1) == "%.0f" % (total * 180 / 8 * 4)
    out2, _ = log(2 * G, x["alloc_ue"][:2 * G], x["alloc_rbg"][:2 * G])
    assert _parse_users(out2) != want

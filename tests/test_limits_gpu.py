"""Every scheduler id at the limits rs_create accepts, against the CPU oracle, bit for bit.

The other parity tests stay well inside the limits (at most ~32 slices for most ids, a few hundred UEs).  Here:

a. UpperBound (id 10) past 2G grants.  Every slice with a positive quota takes its own best min(quota, G) RBGs, so
   a TTI can make up to S*G grants; with many slices more than 2G are common.  Each case first asserts from the
   oracle's alloc_n that they occur, then compares every grant (lists of S*G entries), through rs_step, rs_run_host
   in launches of 1, 7 and 64 TTIs, trace replay, finite queues, 512 threads and two bearers.
b. Many slices (33 / 47 / 63 / 64), every id, the bands of 64 / 25 / 16 / 7 RBGs, the three CQI layouts, backlogged
   and queue-aware, uneven slices with 1-UE slices, both CTA widths; three slice profiles of 64 slices.
c. The largest cells: per id and CQI layout, the largest U that rs_create accepts (bisected), for 64 near-equal
   slices and for one giant slice next to 63 one-UE slices.  Two cells x 16 TTIs at that U against the oracle; one
   more UE is refused for shared memory, and the process goes on scheduling correctly.  On an NVIDIA B200 (227 KB of
   shared memory per CTA) this build accepts, for layouts 0 and 1 alike (also in DESIGN.md section 6):
       ids 8 / 9 / 10 / 101 / 103:  5466 (64 near-equal slices), 1223 (giant slice)
       id 1:                        4448, 4448
       ids 7 / 11:                  4429, 479
d. The grant list itself: any length from 2G to S*G is a prefix of the whole list, the default stays 2G and the
   schedule never depends on it.
Plus a bounded seed of tools/fuzz_parity.one_case(limits=True)."""
import numpy as np
import pytest

from radiosaber_b200 import sched
from tests.test_kernel_paths_gpu import IDS, Case, _check_width
from tests.test_profiles_gpu import ProfCase

gpu = pytest.mark.gpu

RS_ERR_UNSUPPORTED = 2
WIDE_MIN_UES = 480   # rs_sched.cu RS_WIDE_MIN_UES


def _ub_case(S, n_rbs, rbg, ups, seed, T=80, **kw):
    """Id 10 on PF slices (epsilon = psi = 1) with Dirichlet(0.5) weights, every bearer listed: the configuration
    whose grants run past 2G soonest.  Both sides list every grant (S*G entries)."""
    c = Case(10, ups, B=4, T=T, seed=seed, n_rbs=n_rbs, rbg=rbg, grant_len=S * (n_rbs // rbg), active=False, **kw)
    c.w = np.random.default_rng(seed + 1).dirichlet(np.ones(S) * 0.5)
    c.p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    if c.hol is not None:
        c.hol = np.abs(c.hol)   # no negative delays: alpha is 0 everywhere
    return c


def _assert_past_2g(c, want):
    n = want[0]["alloc_n"]
    assert (n > 2 * c.G).sum() >= 3, ("the inputs no longer make more than 2G grants", int(n.max()), 2 * c.G)


def _run_step(c, g, bounds):
    """rs_step, one TTI per call (streamed CQI)."""
    outs, states = [], []
    for t in range(c.T):
        kw = {} if c.queue is None else {"queue": c.queue[t], "hol": c.hol[t]}
        outs.append(g.step(c.slabs[t // c.refresh], c.draws[t], dt=float(c.dts[t]), want_aux=True, **kw))
        if t + 1 in bounds:
            states.append(g.get_state())
    return {k: np.stack([x[k] for x in outs]) for k in outs[0]}, states


# ---- a. UpperBound past 2G grants -----------------------------------------------------------------------------------
# (S, n_rbs, rbg, seed): 100 MHz with 64 and 48 slices, 20 MHz (100 RBs) with 28, 10 MHz (48 RBs) with 40, 3 MHz
# (14 RBs) with 20; seeds whose backlogged runs make more than 2G grants
UB_SHAPES = [(64, 512, 8, 1), (48, 512, 8, 1), (28, 100, 4, 3), (40, 48, 3, 2), (20, 14, 2, 2)]


def _ub_ups(S):
    return [1 + (s % 3 == 0) for s in range(S)]


@gpu
@pytest.mark.parametrize("S,n_rbs,rbg,seed", UB_SHAPES)
def test_upperbound_past_2g_step_and_launches(S, n_rbs, rbg, seed):
    c = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed)
    bounds = [70, 80]
    want = c.oracle(bounds)
    _assert_past_2g(c, want)
    g = c.scheduler()
    assert g.grant_list_len == S * c.G
    c.check(_run_step(c, g, bounds), want, tag="step")
    for tpl in (1, 7, 64):
        g.reset_state()
        c.check(c.run_host(g, bounds, tpl), want, tag=f"ttis_per_launch {tpl}")
    g.close()


@gpu
@pytest.mark.parametrize("S,n_rbs,rbg,seed", UB_SHAPES)
def test_upperbound_past_2g_trace_replay(S, n_rbs, rbg, seed):
    c = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed, trace=True)
    bounds = [50, 80]
    want = c.oracle(bounds)
    _assert_past_2g(c, want)
    g = c.scheduler()
    c.check(c.run_host(g, bounds, 16), want, tag="trace")
    g.reset_state()
    c.check(c.run_device(g, bounds, 16), want, tag="trace, device")
    g.close()


@gpu
@pytest.mark.parametrize("S,n_rbs,rbg,seed", [(64, 512, 8, 1), (40, 48, 3, 2)])
def test_upperbound_past_2g_finite_queues(S, n_rbs, rbg, seed):
    c = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed, queue=True)
    bounds = [40, 80]
    want = c.oracle(bounds)
    _assert_past_2g(c, want)
    for tpl in (1, 7, 64):
        g = c.scheduler()
        c.check(c.run_host(g, bounds, tpl), want, tag=f"queues, ttis_per_launch {tpl}")
        g.close()
    g = c.scheduler()
    c.check(c.run_device(g, bounds, 7), want, tag="queues, device")
    g.close()


@gpu
def test_upperbound_past_2g_wide():
    """64 slices x 8 UEs: 512 threads."""
    c = _ub_case(64, 512, 8, [8] * 64, 11, T=60)
    bounds = [30, 60]
    want = c.oracle(bounds)
    _assert_past_2g(c, want)
    g = c.scheduler()
    _check_width(g, "wide")
    c.check(c.run_host(g, bounds, 16), want)
    g.close()


@gpu
@pytest.mark.parametrize("S,n_rbs,rbg,seed", [(64, 512, 8, 1), (40, 48, 3, 2)])
def test_upperbound_past_2g_two_bearers(S, n_rbs, rbg, seed):
    c = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed, T=60, nb=2)
    bounds = [30, 60]
    want = c.oracle(bounds)
    _assert_past_2g(c, want)
    g = c.scheduler()
    c.check(c.run_host(g, bounds, 7), want)
    g.close()


# ---- d. the grant list at every length ------------------------------------------------------------------------------
@gpu
def test_grant_list_length_prefix_and_default():
    """The default list is 2G (what callers that never set it allocate); lengths 2G..S*G return a prefix of the whole
    list and the same schedule; lengths outside the range and ids other than 10 are refused."""
    S, n_rbs, rbg, seed = 40, 48, 3, 2
    full = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed, T=40)
    bounds = [25, 40]
    want = full.oracle(bounds)
    _assert_past_2g(full, want)
    G = full.G
    assert sched.lib().rs_abi_version() == 3
    for L in (None, 2 * G + 1, 3 * G, S * G - 1, S * G):
        c = _ub_case(S, n_rbs, rbg, _ub_ups(S), seed, T=40)
        c.grant_len = L
        g = c.scheduler()
        n = 2 * G if L is None else L
        assert g.grant_list_len == n
        got = c.run_host(g, bounds, 7)
        assert got[0]["alloc_ue"].shape[-1] == n
        cut = ({k: (v[..., :n] if k in ("alloc_ue", "alloc_rbg") else v) for k, v in want[0].items()}, want[1])
        c.check(got, cut, tag=f"list length {n}")
        g.close()
    g = full.scheduler()
    for bad in (2 * G - 1, S * G + 1, 0, -1):
        with pytest.raises(sched.RsError, match="rs_set_grant_list_len"):
            g.set_grant_list_len(bad)
    assert g.grant_list_len == S * G
    g.close()
    g9 = sched.Scheduler(9, full.w, full.p, full.u2s, 2, n_rbs=n_rbs, rbg_size=rbg)
    assert g9.grant_list_len == 0
    with pytest.raises(sched.RsError, match="id 10"):
        g9.set_grant_list_len(2 * G)
    g9.close()


# ---- b. many slices, every id ----------------------------------------------------------------------------------------
MANY_S = (33, 47, 63)
MANY_BANDS = [(512, 8), (100, 4), (48, 3), (14, 2)]   # 64, 25, 16 and 7 RBGs


def _uneven(S, width):
    """Uneven slices with a 1-UE slice every fourth: ~2 UEs per slice (128 threads), or >= 480 UEs (512 threads)."""
    if width == "narrow":
        return [1 if s % 4 == 0 else 1 + s % 5 for s in range(S)]
    big = -(-600 // (S - (S + 3) // 4))
    return [1 if s % 4 == 0 else big - s % 3 for s in range(S)]


def _many_cases():
    """Per id: S = 64 on 64 RBGs on both widths, then S = 33 / 47 / 63 on rotating bands, layouts and widths."""
    out = []
    for i, algo in enumerate(IDS):
        out += [(algo, 64, MANY_BANDS[0], w, i % 3, i % 2 == 0) for w in ("narrow", "wide")]
        for k, S in enumerate(MANY_S):
            band = MANY_BANDS[(i + k + 1) % 4]
            layout = (i + k) % 3
            if layout == 2 and (band[0] // band[1]) % 8:
                layout = 0
            out.append((algo, S, band, ("narrow", "wide")[(i + k) % 2], layout, (i + k) % 2 == 1))
    return out


@gpu
@pytest.mark.parametrize("algo,S,band,width,layout,queue", _many_cases())
def test_many_slices(algo, S, band, width, layout, queue):
    """60 TTIs in launches of 16 (state compared at both call boundaries)."""
    n_rbs, rbg = band
    ups = _uneven(S, width)
    assert (sum(ups) >= WIDE_MIN_UES) == (width == "wide")
    G = n_rbs // rbg
    c = Case(algo, ups, B=3, T=60, seed=31 * algo + S + n_rbs + layout + 7 * queue, n_rbs=n_rbs, rbg=rbg, layout=layout,
             queue=queue, grant_len=S * G if algo == 10 else None)
    g = c.scheduler()
    _check_width(g, width)
    bounds = [32, 60]
    c.check(c.run_host(g, bounds, 16), c.oracle(bounds), tag=(algo, S, G, width, layout, queue))
    g.close()


def test_many_slices_grid_covers_every_id_at_64x64_on_both_widths():
    """CPU: the grid of test_many_slices meets S = 64 and G = 64 with every id on both widths, every S, band and layout."""
    grid = _many_cases()
    for algo in IDS:
        assert {w for a, S, band, w, _, _ in grid if a == algo and S == 64 and band == (512, 8)} == {"narrow", "wide"}
    assert {S for _, S, _, _, _, _ in grid} == set(MANY_S) | {64}
    assert {b for _, _, b, _, _, _ in grid} == set(MANY_BANDS)
    assert {l for *_, l, _ in grid} == {0, 1, 2} and {q for *_, q in grid} == {False, True}


@gpu
@pytest.mark.parametrize("algo", [9, 10])
def test_three_profiles_of_64_slices(algo):
    """from_profiles with 3 profiles of 64 slices (uneven, 1-UE slices, same U) on 64 RBGs, 60 TTIs."""
    base = _uneven(64, "narrow")
    rot = base[1:] + base[:1]
    rev = base[::-1]
    c = ProfCase(algo, [base, rot, rev], [0, 1, 2, 2, 1, 0], T=60, seed=77 + algo, queue=True)
    g = c.scheduler()
    assert sched.lib().rs_n_profiles(g._h) == 3
    _check_width(g, "narrow")
    bounds = [40, 60]
    c.check(c.run_host(g, bounds, 16), c.oracle(bounds))
    g.close()


# ---- c. the largest cells --------------------------------------------------------------------------------------------
def _shape_ups(shape, U):
    if shape == "equal":   # 64 slices whose sizes differ by at most one
        return [U // 64 + (s < U % 64) for s in range(64)]
    return [U - 63] + [1] * 63   # one giant slice next to 63 one-UE slices


def _create(algo, ups, layout):
    """A 2-cell handle of this shape, or the RsError rs_create returns."""
    S = len(ups)
    u2s = np.repeat(np.arange(S), ups).astype(np.int32)
    w = np.full(S, 1.0 / S)
    p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
    try:
        return sched.Scheduler(algo, w, p, u2s, 2, cqi_per_rb=layout)
    except sched.RsError as e:
        return e


def _u_max(algo, shape, layout):
    lo, hi = 64, 32768   # lo accepted, hi refused
    g = _create(algo, _shape_ups(shape, lo), layout)
    assert not isinstance(g, sched.RsError), g
    g.close()
    while hi - lo > 1:
        mid = (lo + hi) // 2
        g = _create(algo, _shape_ups(shape, mid), layout)
        if isinstance(g, sched.RsError):
            hi = mid
        else:
            g.close()
            lo = mid
    return lo


@gpu
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("shape", ["equal", "giant"])
@pytest.mark.parametrize("algo", IDS)
def test_largest_cell(algo, shape, layout):
    u_max = _u_max(algo, shape, layout)
    print(f"U_max id {algo} {shape} layout {layout}: {u_max}")
    err = _create(algo, _shape_ups(shape, u_max + 1), layout)
    assert isinstance(err, sched.RsError), u_max
    assert f"rs error {RS_ERR_UNSUPPORTED}" in str(err) and "shared memory" in str(err), str(err)
    ups = _shape_ups(shape, u_max)
    c = Case(algo, ups, B=2, T=16, seed=13 * algo + 5 * layout + (shape == "giant"), layout=layout, active=False,
             refresh=8, grant_len=64 * 64 if algo == 10 else None)
    g = c.scheduler()
    _check_width(g, "wide" if u_max >= WIDE_MIN_UES else "narrow")
    bounds = [8, 16]
    c.check(c.run_host(g, bounds, 8), c.oracle(bounds), tag=("U_max", u_max))
    g.close()
    # the refusal left nothing behind: a small handle created afterwards schedules correctly
    small = Case(algo, [3, 1, 7, 2, 5], B=2, T=6, seed=algo, layout=layout, queue=True)
    g = small.scheduler()
    small.check(small.run_host(g, [6], 3), small.oracle([6]))
    g.close()


@gpu
def test_ue_count_bounds():
    """rs_create: n_ues 32768 is outside 1..32767 (user ids are int16); 32767 is within it but needs more shared memory
    than one CTA has."""
    for U, what in ((32768, "outside 1..32767"), (32767, "shared memory")):
        err = _create(9, _shape_ups("equal", U), 0)
        assert isinstance(err, sched.RsError) and f"rs error {RS_ERR_UNSUPPORTED}" in str(err) and what in str(err), err


# ---- the fuzz near the limits ----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("seed", [2101, 2202])
def test_limits_fuzz(seed):
    """tools/fuzz_parity.one_case(limits=True): every id, 24..64 slices, the bands, up to a few thousand UEs."""
    from tools import fuzz_parity
    rng = np.random.default_rng(seed)
    for case in range(3):
        err = fuzz_parity.one_case(rng, case, limits=True)
        assert err is None, err

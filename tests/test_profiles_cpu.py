"""CPU: rs_create_profiles rejects bad slice profiles before it touches a GPU (the checks run on the host first, so
these pass on a machine without one)."""
import numpy as np
import pytest

from radiosaber_b200 import sched

S, U, B = 3, 6, 5


def _profiles(n=3):
    out = []
    for k in range(n):
        w = np.full(S, 1 / S) + 0.01 * k
        p = np.tile(np.array([0, 0, 1, 1], dtype=np.int32), (S, 1))
        p[:, 2] = k % 3
        u2s = np.array([0, 0, 1, 1, 2, 2], dtype=np.int32) if k % 2 == 0 else np.array([0, 1, 1, 1, 2, 2], dtype=np.int32)
        out.append((w, p, u2s))
    return out


def _create(profiles, cell_profile, n_cells=B, **kw):
    return sched.Scheduler.from_profiles(9, profiles, cell_profile, n_cells=n_cells, **kw)


@pytest.mark.parametrize("field,value", [("algo", 8), ("n_slices", 4), ("n_ues", 7), ("n_rbs", 256), ("rbg_size", 4),
                                         ("cqi_per_rb", 2), ("data_to_transmit", 5000), ("n_bearers", 2),
                                         ("tbs_row_m1", 1)])
def test_shared_field_that_differs_is_named(field, value):
    prof = _profiles()
    sched.lib()
    cfgs = (sched._Cfg * 3)()
    keep = []
    for i, (w, p, m) in enumerate(prof):
        w2, p2, m2 = w, p, m
        if i == 2 and field == "n_slices":
            w2, p2 = np.append(w, 0.1), np.vstack([p, p[:1]])
        if i == 2 and field == "n_ues":
            m2 = np.append(m, 2).astype(np.int32)
        row = None
        if field == "tbs_row_m1" and i == 2:
            row = np.arange(27, dtype=np.int32)
        keep += [w2, p2, m2, row]
        cfgs[i] = sched._Cfg(9, len(w2), len(m2), 512, 8, 0, 100000000, 1, sched._ptr(w2), sched._ptr(p2),
                             sched._ptr(m2), sched._ptr(row))
        if i == 2 and field not in ("n_slices", "n_ues", "tbs_row_m1"):
            setattr(cfgs[i], field, value)
    cp = np.array([0, 1, 2, 1, 0], dtype=np.int32)
    h = sched.C.c_void_p()
    rc = sched.lib().rs_create_profiles(cfgs, 3, sched._ptr(cp), B, 0, sched.C.byref(h))
    msg = sched.lib().rs_last_error().decode()
    assert rc == 1, (rc, msg)
    assert field in msg and "profile 2" in msg, msg


def test_stock_tbs_row_given_explicitly_is_the_same_field():
    """tbs_row_m1 is compared by value: NULL in one profile and the stock row spelled out in another agree (the
    call then only fails for want of a GPU, or succeeds on one)."""
    mcs_to_itbs = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 15, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26]
    stock = np.array([mcs_to_itbs[i + 5] if i + 5 < 29 else 0 for i in range(27)], dtype=np.int32)
    prof = _profiles(2)
    cfgs = (sched._Cfg * 2)()
    keep = []
    for i, (w, p, m) in enumerate(prof):
        row = stock if i == 1 else None
        keep.append(row)
        cfgs[i] = sched._Cfg(9, S, U, 512, 8, 0, 100000000, 1, sched._ptr(w), sched._ptr(p), sched._ptr(m), sched._ptr(row))
    cp = np.array([0, 1, 1, 0, 1], dtype=np.int32)
    h = sched.C.c_void_p()
    rc = sched.lib().rs_create_profiles(cfgs, 2, sched._ptr(cp), B, 0, sched.C.byref(h))
    msg = sched.lib().rs_last_error().decode()
    assert "tbs_row_m1" not in msg
    if rc == 0:
        sched.lib().rs_destroy(h)
    else:
        assert rc == 3, (rc, msg)   # no GPU here: every argument check passed


def test_psi_out_of_range_names_psi_and_the_profile():
    prof = _profiles()
    prof[2][1][1, 3] = 2
    with pytest.raises(sched.RsError, match=r"profile 2: slice 1: psi=2"):
        _create(prof, [0, 1, 2, 0, 1])


def test_ue_to_slice_out_of_range_names_the_profile():
    prof = _profiles()
    prof[1][2][4] = S
    with pytest.raises(sched.RsError, match=r"rs error 1: profile 1: ue_to_slice\[4\] out of range"):
        _create(prof, [0, 1, 2, 0, 1])


def test_cell_profile_out_of_range_or_missing():
    prof = _profiles()
    with pytest.raises(sched.RsError, match=r"cell_profile\[3\] = 3 outside 0..2"):
        _create(prof, [0, 1, 2, 3, 1])
    with pytest.raises(sched.RsError, match=r"cell_profile\[0\] = -1"):
        _create(prof, [-1, 1, 2, 0, 1])
    with pytest.raises(sched.RsError, match="cell_profile is NULL with 3 profiles"):
        _create(prof, None)


def test_profile_count_outside_one_to_n_cells():
    prof = _profiles()
    with pytest.raises(sched.RsError, match="n_profiles 0 outside"):
        sched.Scheduler(9, *prof[0], B, profiles=[], cell_profile=[0] * B)
    with pytest.raises(sched.RsError, match="n_profiles 3 outside 1..n_cells \\(2\\)"):
        _create(prof, [0, 1], n_cells=2)


def test_per_profile_checks_of_rs_create_run_on_every_profile():
    """Id 7's required-RBs guard and id 1's flow-satisfied cut-off are checks of shared fields; the profile checks
    (psi, ue_to_slice) run on every profile, not only on profile 0."""
    prof = _profiles()
    prof[0][1][0, 3] = 0
    prof[1][1][2, 3] = 7
    with pytest.raises(sched.RsError, match="profile 1: slice 2: psi=7"):
        _create(prof, [0, 1, 2, 0, 1])
    with pytest.raises(sched.RsError, match="required-RBs guard"):
        sched.Scheduler.from_profiles(7, _profiles(), [0, 1, 2, 0, 1], data_to_transmit=5000)
    with pytest.raises(sched.RsError, match="flow-satisfied"):
        sched.Scheduler.from_profiles(1, _profiles(), [0, 1, 2, 0, 1], data_to_transmit=10)


def test_one_profile_keeps_the_messages_of_rs_create():
    prof = _profiles(1)
    prof[0][1][1, 3] = 2
    with pytest.raises(sched.RsError, match=r"rs error 2: slice 1: psi=2"):
        _create(prof, None)

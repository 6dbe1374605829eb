"""CPU: the per-bearer FIFO model (tests/buffer_model.py) on hand-computed numbers, and the synthetic-arrival generator
(workload.synth_arrivals, twin of rs_synth_arrivals).  The device path is checked against both in test_buffers_gpu.py."""
import numpy as np
import pytest

from radiosaber_b200 import sched, workload
from tests.buffer_model import INFINITE, BufferModel


def test_arrival_then_shown_queue_and_delay():
    m = BufferModel((1, 2), 3)
    q, h = m.arrive([[500, 0]], now=1.0, arrival_time=0.9996)
    assert q.tolist() == [[500, 0]] and h[0, 0] == 1.0 - 0.9996 and h[0, 1] == 0.0
    q, h = m.arrive([[0, -5]], now=1.001, arrival_time=1.0)        # nothing arrives; the delay grows
    assert q.tolist() == [[500, 0]] and h[0, 0] == 1.001 - 0.9996


def test_partial_send_keeps_the_head_timestamp():
    m = BufferModel((1,), 4)
    m.arrive([300], 1.0, 0.5)
    m.arrive([200], 1.001, 0.9)
    m.depart([120])
    st = m.state()
    assert st["queued"][0] == 380 and st["n_records"][0] == 2 and st["head_time"][0] == 0.5
    m.depart([180])                      # exactly the rest of the head: popped
    st = m.state()
    assert st["queued"][0] == 200 and st["n_records"][0] == 1 and st["head_time"][0] == 0.9
    q, h = m.arrive([0], 1.002, 1.002)
    assert q[0] == 200 and h[0] == 1.002 - 0.9


def test_departure_is_clamped_to_the_queue():
    m = BufferModel((1,), 4)
    m.arrive([10], 1.0, 1.0)
    m.depart([4000])                     # id 1 books its whole TBS
    st = m.state()
    assert st["queued"][0] == 0 and st["n_records"][0] == 0 and st["head_time"][0] == 0.0
    assert m.arrive([0], 1.001, 1.001)[0][0] == 0


def test_overflow_drops_whole_arrivals():
    m = BufferModel((1,), 2)
    for t, a in enumerate((100, 200, 300, 7)):
        m.arrive([a], 1.0 + t * 0.001, 1.0 + t * 0.001)
    st = m.state()
    assert st["queued"][0] == 300 and st["n_records"][0] == 2 and st["dropped"][0] == 307
    m.depart([100])
    m.arrive([50], 1.004, 1.004)         # room again
    assert m.state()["queued"][0] == 250 and m.state()["dropped"][0] == 307


def test_backlogged_bearers_have_no_fifo():
    m = BufferModel((1, 2), 2, backlogged=[[True, False]])
    q, h = m.arrive([[900, 900]], 1.0, 0.9)
    assert q.tolist() == [[INFINITE, 900]] and h[0, 0] == 0.0
    m.depart([[5000, 100]])
    st = m.state()
    assert st["queued"].tolist() == [[0, 800]] and st["n_records"].tolist() == [[0, 1]]


def test_queue_shown_saturates_at_int32():
    m = BufferModel((1,), 2)
    m.arrive([2_000_000_000], 1.0, 1.0)
    q, _ = m.arrive([2_000_000_000], 1.001, 1.001)
    assert q[0] == 2147483647 and m.state()["queued"][0] == 4_000_000_000


def test_synth_arrivals_rule_and_determinism():
    u2s = np.array([0, 0, 1, 1, 2], np.int32)
    pkt = np.array([100, 0, 1500], np.int32)
    q16 = np.array([int(2.25 * 65536), 5 * 65536, 3 * 65536], np.int32)
    a = workload.synth_arrivals(7, 3, 4, 10, 50, u2s, pkt, q16)
    assert a.shape == (50, 4, 5) and a.dtype == np.int32
    assert set(np.unique(a[:, :, :2])) == {200, 300}          # 2 or 3 packets of 100 B, a quarter of the TTIs 3
    assert 0.15 < (a[:, :, :2] == 300).mean() < 0.35
    assert (a[:, :, 2:4] == 0).all() and (a[:, :, 4] == 4500).all()
    assert np.array_equal(a, workload.synth_arrivals(7, 3, 4, 10, 50, u2s, pkt, q16))
    # any (cell, tti) shard is the same slice of the whole
    part = workload.synth_arrivals(7, 5, 2, 30, 20, u2s, pkt, q16)
    assert np.array_equal(part, a[20:40, 2:4])
    assert not np.array_equal(a, workload.synth_arrivals(8, 3, 4, 10, 50, u2s, pkt, q16))
    two = workload.synth_arrivals(7, 3, 4, 10, 50, u2s, pkt, q16, n_bearers=2)
    assert two.shape == (50, 4, 5, 2) and np.array_equal(two[..., 0], a)
    # profiles: cell b reads its profile's row
    prof = workload.synth_arrivals(7, 3, 4, 10, 50, np.stack([u2s, u2s]), np.stack([pkt, pkt * 0]),
                                   np.stack([q16, q16]), cell_profile=[0, 1, 0, 1])
    assert np.array_equal(prof[:, [0, 2]], a[:, [0, 2]]) and (prof[:, [1, 3]] == 0).all()


def test_buffer_calls_refuse_bad_arguments_without_a_gpu():
    """The host-side checks that need no device: a null handle."""
    L = sched.lib()
    assert L.rs_enable_buffers(None, 4, None) == 1
    assert L.rs_set_traffic(None, None) == 1
    assert L.rs_get_buffers(None, None, None, None, None) == 1
    assert L.rs_synth_arrivals(None, 0, 0, 0, 1, None, None, None) == 1

"""Synthetic workload of SURVEY.md section 8(d): counter-based CQI / rand() streams.

CQI is i.i.d. from the empirical histogram of the reference's
``cqi-traces-noise0`` traces (4 803 200 samples, values 1..15), one value per
(cell, tti // refresh, ue, rbg) -- every RBG's RBs share the value, exactly the
structure of the shipped traces (enb-mac-entity.cc:160-193 feeds them in).
The generator is ``splitmix64`` of a packed counter so that any shard of the
(cell, tti) space can be produced independently on any rank or device
(``rs_synth_cqi`` in the C ABI is the device twin of :func:`synth_cqi`).
"""
from __future__ import annotations

import numpy as np

# counts of CQI 1..15 over all 158 traces (SURVEY.md section 8(d))
CQI_HIST = np.array([19075, 7082, 33860, 261099, 438688, 199446, 518174, 661977, 237928, 861279,
                     596358, 355319, 447453, 12000, 153462], dtype=np.uint64)
CQI_TOTAL = int(CQI_HIST.sum())
# thresholds on a 32-bit uniform: cqi = 1 + #{k : u32 >= CQI_CDF32[k]}, k = 0..13
CQI_CDF32 = ((np.cumsum(CQI_HIST)[:-1].astype(np.float64) / CQI_TOTAL) * 4294967296.0).astype(np.uint64).astype(np.uint32)

_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)
_GOLD = np.uint64(0x9E3779B97F4A7C15)
DOMAIN_CQI = 0x43514900  # "CQI\0"
DOMAIN_RAND = 0x524E4400  # "RND\0"


def splitmix64(x: np.ndarray) -> np.ndarray:
    """Finaliser of splitmix64 applied to ``x + golden`` (uint64, wrapping)."""
    with np.errstate(over="ignore"):
        z = x.astype(np.uint64) + _GOLD
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        return z ^ (z >> np.uint64(31))


def _key(seed: int, domain: int) -> np.uint64:
    return splitmix64(np.array([(seed & 0xFFFFFFFF) | (domain << 32)], dtype=np.uint64))[0]


def synth_cqi(seed: int, cell0: int, n_cells: int, tti0: int, n_ttis: int, n_ues: int, n_rbgs: int,
              refresh: int = 1) -> np.ndarray:
    """uint8 [n_ttis][n_cells][n_ues][n_rbgs] with values 1..15."""
    key = _key(seed, DOMAIN_CQI)
    epoch = (np.arange(tti0, tti0 + n_ttis, dtype=np.uint64) // np.uint64(refresh))[:, None, None, None]
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[None, :, None, None]
    ue = np.arange(n_ues, dtype=np.uint64)[None, None, :, None]
    rbg = np.arange(n_rbgs, dtype=np.uint64)[None, None, None, :]
    with np.errstate(over="ignore"):
        ctr = (epoch << np.uint64(40)) ^ (cell << np.uint64(20)) ^ (ue << np.uint64(8)) ^ rbg
        # ue can exceed 12 bits in the sweep configs: fold the overflow in with a multiply
        ctr = ctr ^ ((ue >> np.uint64(12)) * np.uint64(0xD6E8FEB86659FD93))
        h = splitmix64(ctr ^ key)
    u32 = (h >> np.uint64(32)).astype(np.uint32)
    cqi = np.ones(u32.shape, dtype=np.uint8)
    for thr in CQI_CDF32:
        cqi += (u32 >= thr).astype(np.uint8)
    return cqi


def histogram_cqi(rng: np.random.Generator, shape) -> np.ndarray:
    """uint8 array of the given shape, i.i.d. from the same histogram through a numpy generator (synthetic
    trace files; not the counter-based stream above)."""
    u32 = rng.integers(0, 1 << 32, size=shape, dtype=np.uint64).astype(np.uint32)
    cqi = np.ones(u32.shape, dtype=np.uint8)
    for thr in CQI_CDF32:
        cqi += (u32 >= thr).astype(np.uint8)
    return cqi


def synth_rand2(seed: int, cell0: int, n_cells: int, tti0: int, n_ttis: int, n_slices: int) -> np.ndarray:
    """int32 [n_ttis][n_cells][2]: the two rand() values of transport.cpp:490,511.

    Values lie in [0, 2^31 - 1 - n_slices] so that ``(i + rand) % S`` cannot overflow int
    (SURVEY H5).
    """
    key = _key(seed, DOMAIN_RAND)
    tti = np.arange(tti0, tti0 + n_ttis, dtype=np.uint64)[:, None, None]
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[None, :, None]
    which = np.arange(2, dtype=np.uint64)[None, None, :]
    with np.errstate(over="ignore"):
        ctr = (tti << np.uint64(32)) ^ (cell << np.uint64(1)) ^ which
        h = splitmix64(ctr ^ key)
    span = np.uint64(2147483647 - n_slices + 1)
    return ((h >> np.uint64(11)) % span).astype(np.int32)


def synth_rand_draws(seed: int, cell0: int, n_cells: int, tti0: int, n_ttis: int, n_slices: int, stride: int) -> np.ndarray:
    """int32 [n_ttis][n_cells][stride]: the rand() values a scheduler draws per cell-TTI.  stride 2 is
    :func:`synth_rand2`; wider strides (id 11: 300 x the largest slice, downlink-nvs-scheduler.cpp:437-446)
    pack the counter differently.  Twin of ``rs_synth_rand2`` in the C ABI."""
    if stride == 2:
        return synth_rand2(seed, cell0, n_cells, tti0, n_ttis, n_slices)
    key = _key(seed, DOMAIN_RAND)
    tti = np.arange(tti0, tti0 + n_ttis, dtype=np.uint64)[:, None, None]
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[None, :, None]
    which = np.arange(stride, dtype=np.uint64)[None, None, :]
    with np.errstate(over="ignore"):
        ctr = (tti << np.uint64(40)) ^ (cell << np.uint64(16)) ^ which ^ np.uint64(0x5EA4C4000000)
        h = splitmix64(ctr ^ key)
    span = np.uint64(2147483647 - n_slices + 1)
    return ((h >> np.uint64(11)) % span).astype(np.int32)


def tti_clock(n_ttis: int, start: float = 0.1):
    """The reference's TTI clock: FrameManager re-schedules itself every 0.001 s and the
    simulator accumulates ``t += 0.001`` in double (simulator.cc:116-126), applications start at
    ``start`` (single-cell-with-interference.h:254).  Returns (now[n_ttis], dt[n_ttis]) for the
    first n_ttis TTIs that have bearers; dt[0] = now[0] - start is what the first EWMA update
    sees (RadioBearer's lastUpdate is its creation time, radio-bearer.cpp:54-55,131-136).
    """
    t = 0.0
    while t < start:
        t = t + 0.001
    now = np.empty(n_ttis, dtype=np.float64)
    dt = np.empty(n_ttis, dtype=np.float64)
    last = start
    for k in range(n_ttis):
        now[k] = t
        dt[k] = t - last
        last = t
        t = t + 0.001
    return now, dt


DOMAIN_ARRIVALS = 0x41525200  # "ARR\0"


def synth_arrivals(seed: int, cell0: int, n_cells: int, tti0: int, n_ttis: int, ue_to_slice, pkt_bytes, pkts_q16,
                   n_bearers: int = 1, cell_profile=None) -> np.ndarray:
    """int32 [n_ttis][n_cells][U] ([..][U][2] with two bearers): bytes arriving at each bearer per TTI, for the
    device-kept buffers (``rs_enable_buffers``; ``rs_synth_arrivals`` is the device twin).

    ue_to_slice [U] or [P][U], pkt_bytes / pkts_q16 [S] or [P][S] (one row per slice profile; cell b reads row
    cell_profile[b], row 0 without profiles).  A bearer of slice s gets ``(q >> 16) + (draw16 < (q & 0xffff))``
    packets of ``pkt_bytes[s]`` bytes with ``q = pkts_q16[s]`` (packets per TTI in 16.16 fixed point); draw16 is the
    top 16 bits of one splitmix64 draw of a counter over (cell, tti, ue, slot) built like :func:`synth_cqi`'s.
    Integers only, so the two twins agree bit for bit."""
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    pb = np.atleast_2d(np.asarray(pkt_bytes, dtype=np.int64))
    pq = np.atleast_2d(np.asarray(pkts_q16, dtype=np.int64))
    U = u2s.shape[1]
    nb = 2 if int(n_bearers) == 2 else 1
    cp = np.zeros(n_cells, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)
    key = _key(seed, DOMAIN_ARRIVALS)
    tti = np.arange(tti0, tti0 + n_ttis, dtype=np.uint64)[:, None, None, None]
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[None, :, None, None]
    ue = np.arange(U, dtype=np.uint64)[None, None, :, None]
    slot = np.arange(nb, dtype=np.uint64)[None, None, None, :]
    with np.errstate(over="ignore"):
        ctr = ((tti << np.uint64(40)) ^ (cell << np.uint64(20)) ^ (ue << np.uint64(8)) ^ slot)
        ctr = ctr ^ ((ue >> np.uint64(12)) * np.uint64(0xD6E8FEB86659FD93))
        draw16 = (splitmix64(ctr ^ key) >> np.uint64(48)).astype(np.int64)
    s = u2s[cp]                                            # [B][U]: each cell's slices
    size = np.take_along_axis(pb[cp], s, axis=1)[None, :, :, None]
    q = np.take_along_axis(pq[cp], s, axis=1)[None, :, :, None]
    out = (size * ((q >> 16) + (draw16 < (q & 0xffff)))).astype(np.int32)
    return out if nb == 2 else out[..., 0]

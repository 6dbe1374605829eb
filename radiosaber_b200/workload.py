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


DOMAIN_SOURCES = 0x53524300  # "SRC\0"
SRC_NONE, SRC_RATE, SRC_PERIODIC, SRC_ONOFF = 0, 1, 2, 3


def synth_traffic(seed: int, cell0: int, n_cells: int, tti0: int, n_ttis: int, ue_to_slice, sources, n_bearers: int = 1,
                  cell_profile=None, state=None):
    """(arrivals, state): int32 [n_ttis][n_cells][U] ([..][U][2] with two bearers) bytes arriving at each bearer from the
    traffic sources, and the on-off chains after the last TTI (uint8, shaped like one TTI of arrivals, 1 = ON; 0 for
    bearers of other kinds).  ``rs_set_sources`` + ``rs_synth_traffic`` is the device twin, bit for bit.

    sources: one dict per slice ([S]), or one list per slice profile ([P][S]), with the fields of ``rs_source``:
    ``kind`` (SRC_NONE / SRC_RATE / SRC_PERIODIC / SRC_ONOFF) and ``pkt_bytes``, ``pkts_q16``, ``period_ttis``,
    ``frame_bytes`` (a list), ``leave_on_q32``, ``leave_off_q32`` as the kind needs them.  state: what an earlier call
    returned, for a call that continues at its tti0 + n_ttis; None = the chains start from their initial draw.  The rules
    are those of include/rs_sched.h: global TTI tau = tti0 + t, global cell = cell0 + b; one draw per (tau, cell, ue, slot)
    (:func:`synth_arrivals`' counter and key: RATE is :func:`synth_arrivals` itself, ONOFF takes the low 32 bits) and one
    per (cell, ue, slot) under key "SRC" without tau (phase, start frame, initial on-off state)."""
    src = [list(sources)] if isinstance(sources[0], dict) else [list(p) for p in sources]
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    P, S, U = len(src), len(src[0]), u2s.shape[1]
    nb = 2 if int(n_bearers) == 2 else 1
    cp = np.zeros(n_cells, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)

    def field(name, default=0):
        return np.array([[int(e.get(name, default)) for e in row] for row in src], dtype=np.int64)   # [P][S]

    kind = field("kind")
    rate = kind == SRC_RATE
    arr = synth_arrivals(seed, cell0, n_cells, tti0, n_ttis, u2s, np.where(rate, field("pkt_bytes"), 0),
                         np.where(rate, field("pkts_q16"), 0), n_bearers=nb, cell_profile=cp)
    arr = arr.reshape(n_ttis, n_cells, U, nb).astype(np.int64)

    def per_bearer(a):   # [P][S] -> [B][U][1]
        return np.take_along_axis(a[cp], u2s[cp], axis=1)[:, :, None]

    k = per_bearer(kind)
    period = per_bearer(np.maximum(field("period_ttis", 1), 1))
    key = _key(seed, DOMAIN_SOURCES)
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[:, None, None]
    ue = np.arange(U, dtype=np.uint64)[None, :, None]
    slot = np.arange(nb, dtype=np.uint64)[None, None, :]
    with np.errstate(over="ignore"):
        ctr = (cell << np.uint64(20)) ^ (ue << np.uint64(8)) ^ slot ^ ((ue >> np.uint64(12)) * np.uint64(0xD6E8FEB86659FD93))
        hb = splitmix64(ctr ^ key)
    lo = (hb & np.uint64(0xFFFFFFFF)).astype(np.int64)                    # [B][U][nb]
    phi = ((hb >> np.uint64(32)) % period.astype(np.uint64)).astype(np.int64)
    tau = np.arange(tti0, tti0 + n_ttis, dtype=np.int64)[:, None, None, None]
    x = tau + phi                                                          # [T][B][U][nb]
    aligned = x % period == 0

    periodic = k == SRC_PERIODIC
    if periodic.any():
        frames = [np.asarray(e.get("frame_bytes", [1]), dtype=np.int64) if e["kind"] == SRC_PERIODIC else np.ones(1, np.int64)
                  for row in src for e in row]
        n_frames = np.array([len(f) for f in frames], dtype=np.int64).reshape(P, S)
        offset = np.concatenate([[0], np.cumsum(n_frames.reshape(-1))[:-1]]).reshape(P, S)
        nf, off = per_bearer(n_frames), per_bearer(offset)
        fi = (x // period + lo % nf) % nf
        size = np.concatenate(frames)[off + fi]
        arr = np.where(periodic & aligned, size, arr)

    on = np.zeros((n_cells, U, nb), dtype=bool)
    onoff = k == SRC_ONOFF
    if onoff.any():
        leave_on, leave_off = per_bearer(field("leave_on_q32")), per_bearer(field("leave_off_q32"))
        if state is None:
            # the stationary ON probability leave_off / (leave_on + leave_off) in 0.32 fixed point, rounded down
            thr = (leave_off.astype(np.uint64) << np.uint64(32)) // np.maximum(leave_on + leave_off, 1).astype(np.uint64)
            on = lo < thr.astype(np.int64)
        else:
            on = np.asarray(state).reshape(n_cells, U, nb) != 0
        on &= onoff
        pkt = per_bearer(field("pkt_bytes"))
        akey = _key(seed, DOMAIN_ARRIVALS)
        with np.errstate(over="ignore"):
            for t in range(n_ttis):
                draw = (splitmix64((np.uint64(tti0 + t) << np.uint64(40)) ^ ctr ^ akey) & np.uint64(0xFFFFFFFF)).astype(np.int64)
                on ^= onoff & (draw < np.where(on, leave_on, leave_off))
                arr[t] = np.where(onoff, np.where(on & aligned[t], pkt, 0), arr[t])
    out, st = arr.astype(np.int32), on.astype(np.uint8)
    return (out, st) if nb == 2 else (out[..., 0], st[..., 0])


DOMAIN_CHANNEL = 0x43484E00  # "CHN\0"
CH_IID, CH_FADING = 0, 1
N_PATHS = 8
_FOLD = np.uint64(0xD6E8FEB86659FD93)
_M32 = np.uint64(0xFFFFFFFF)


def cos_q14() -> np.ndarray:
    """int16 [1024]: round(16384 cos(2 pi i / 1024)), the channel's cosine table (include/rs_cos_q14.inc is written
    from this by tools/gen_cos_table.py)."""
    i = np.arange(1024, dtype=np.float64)
    return np.round(16384.0 * np.cos(2.0 * np.pi * i / 1024.0)).astype(np.int16)


def _slope(raw, coherence):
    """uint64 phase slopes uniform over [-W, W] mod 2^32, W = floor(2^31 / coherence) (0 for coherence 0)."""
    coh = np.asarray(coherence, dtype=np.int64)
    w = np.where(coh > 0, (1 << 31) // np.maximum(coh, 1), 0).astype(np.uint64)
    return (((raw * (np.uint64(2) * w + np.uint64(1))) >> np.uint64(32)) - w) & _M32


def _channel_paths(seed, cell0, n_cells, n_ues, coherence_rbgs, coherence_epochs):
    """The per-(cell, UE) draws of a FADING channel: level draw uint64 [B][U] and theta, omega, nu uint64 [B][U][8]."""
    key = _key(seed, DOMAIN_CHANNEL)
    cell = np.arange(cell0, cell0 + n_cells, dtype=np.uint64)[:, None, None]
    ue = np.arange(n_ues, dtype=np.uint64)[None, :, None]
    idx = np.arange(1 + 2 * N_PATHS, dtype=np.uint64)[None, None, :]
    with np.errstate(over="ignore"):
        ctr = (cell << np.uint64(20)) ^ (ue << np.uint64(8)) ^ idx ^ ((ue >> np.uint64(12)) * _FOLD)
        h = splitmix64(ctr ^ key)                                 # [B][U][17]
    hi, lo = h >> np.uint64(32), h & _M32
    shape = (n_cells, n_ues, 1)
    omega = _slope(lo[..., 1:1 + N_PATHS], np.broadcast_to(np.asarray(coherence_rbgs), (n_cells, n_ues)).reshape(shape))
    nu = _slope(hi[..., 1 + N_PATHS:], np.broadcast_to(np.asarray(coherence_epochs), (n_cells, n_ues)).reshape(shape))
    return hi[..., 0], hi[..., 1:1 + N_PATHS], omega, nu


def _offset_sum(theta, omega, nu, epoch0, n_epochs, n_rbgs):
    tab = cos_q14().astype(np.int64)
    g = np.arange(n_rbgs, dtype=np.uint64)
    e = (np.arange(epoch0, epoch0 + n_epochs, dtype=np.int64) & 0xFFFFFFFF).astype(np.uint64)[:, None, None, None]
    x = np.zeros((n_epochs,) + theta.shape[:2] + (n_rbgs,), dtype=np.int64)
    for k in range(N_PATHS):
        ph = (theta[None, :, :, k, None] + g * omega[None, :, :, k, None] + e * nu[None, :, :, k, None]) & _M32
        x += tab[(ph >> np.uint64(22)).astype(np.intp)]
    return x


def channel_offset_sum(seed, cell0, n_cells, epoch0, n_epochs, n_ues, n_rbgs, coherence_rbgs, coherence_epochs):
    """int64 [E][B][U][G]: the FADING channel's sum x of eight Q14 cosines before depth, rounding and clamping (standard
    deviation 2^15; autocorrelation sinc(pi dg / coherence_rbgs) x sinc(pi de / coherence_epochs)).  The coherences are
    scalars or [B][U]; x does not depend on the level or the depth.  For the statistical tests."""
    _, th, om, nu = _channel_paths(seed, cell0, n_cells, n_ues, coherence_rbgs, coherence_epochs)
    return _offset_sum(th, om, nu, epoch0, n_epochs, n_rbgs)


def synth_channel(seed: int, cell0: int, n_cells: int, epoch0: int, n_epochs: int, ue_to_slice, channels,
                  cell_profile=None, n_rbgs: int = 64) -> np.ndarray:
    """uint8 [n_epochs][n_cells][U][n_rbgs], values 1..15: the synthetic channel's CQI of epochs epoch0.. (one value per
    RBG; :func:`radiosaber_b200.sched.pack_cqi` gives layout 2).  ``rs_set_channels`` + ``rs_synth_channel`` is the
    device twin, bit for bit.

    channels: one dict per slice ([S]), or one list per slice profile ([P][S]), with the fields of ``rs_channel``:
    ``kind`` (CH_IID / CH_FADING) and, for FADING, ``level_thr`` (14 ints), ``depth_q8``, ``coherence_rbgs``,
    ``coherence_epochs`` (``sched.channel_spec`` makes them).  ue_to_slice [U] or [P][U]; cell b uses row
    cell_profile[b].  The rules are those of include/rs_sched.h: IID is :func:`synth_cqi` itself; FADING is
    clamp(L + ((x * depth_q8 + 2^22) >> 23), 1, 15) with the per-UE level L and x of :func:`channel_offset_sum`."""
    rows = [list(channels)] if isinstance(channels[0], dict) else [list(p) for p in channels]
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    U = u2s.shape[1]
    cp = np.zeros(n_cells, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)

    def per_ue(a):   # [P][S](...) -> [B][U](...)
        return a[cp[:, None], u2s[cp]]

    def field(name):
        return np.array([[int(e.get(name, 0)) for e in r] for r in rows], dtype=np.int64)

    out = synth_cqi(seed, cell0, n_cells, epoch0, n_epochs, U, n_rbgs)
    fading = per_ue(field("kind")) == CH_FADING
    if not fading.any():
        return out
    thr = per_ue(np.array([[list(e.get("level_thr", [0] * 14)) for e in r] for r in rows], dtype=np.int64))
    lv, th, om, nu = _channel_paths(seed, cell0, n_cells, U, per_ue(field("coherence_rbgs")),
                                    per_ue(field("coherence_epochs")))
    level = 1 + (lv.astype(np.int64)[..., None] >= thr).sum(axis=-1)                    # [B][U]
    x = _offset_sum(th, om, nu, epoch0, n_epochs, n_rbgs)
    off = (x * per_ue(field("depth_q8"))[None, :, :, None] + (1 << 22)) >> 23
    cqi = np.clip(level[None, :, :, None] + off, 1, 15)
    return np.where(fading[None, :, :, None], cqi, out).astype(np.uint8)


def hol_hist(queue, hol, tbs_bits, algo: int, ue_to_slice, backlogged, n_slices: int, n_bins: int,
             bins_per_unit: float = 1000.0, cell_profile=None) -> np.ndarray:
    """uint64 [P][2][S][n_bins]: the head-of-line delay histograms a buffered handle counts with ``rs_enable_hol_hist``
    (the device twin, bit for bit), from what a run showed and sent.

    queue int32 / hol float64 [T][B][U] ([..][U][2] with two bearers): the run's queue_out / hol_out; tbs_bits int32
    [T][B][U]; backlogged bool [B][U] ([B][U][2]): bearers without a FIFO, which add nothing; ue_to_slice [U] or [P][U]
    and cell_profile [B] (None = profile 0): cell b counts in row cell_profile[b] with that profile's slices.
    Row 0 books the bearers that send (``rs_log_tti``'s stderr rule: tbs_bits / 8 bytes go from slot nb-1 down, a slot
    with queue <= 0 skipped except for id 1, until none are left), row 1 every bearer with queue > 0; the bin is
    min(floor(hol * bins_per_unit + 0.5), n_bins - 1), the product and the sum each rounded (numpy does not fuse)."""
    tbs = np.asarray(tbs_bits, dtype=np.int64)
    T, B, U = tbs.shape
    q = np.asarray(queue, dtype=np.int64).reshape(T, B, U, -1)
    h = np.asarray(hol, dtype=np.float64).reshape(q.shape)
    nb = q.shape[3]
    fifo = ~np.asarray(backlogged, dtype=bool).reshape(B, U, nb)
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    P, S = u2s.shape[0], int(n_slices)
    cp = np.zeros(B, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)
    row0 = ((cp * 2)[:, None] * S + u2s[cp]) * n_bins              # [B][U]: [pf][0][s][0]
    d = np.floor(h * float(bins_per_unit) + 0.5)
    bins = np.minimum(d, n_bins - 1).astype(np.int64)
    avail = tbs // 8
    idx, keep = [], []
    for k in range(nb - 1, -1, -1):
        qk = q[..., k]
        served = (avail > 0) & ((qk > 0) | (algo == 1))
        avail = np.where(served, avail - (avail if algo == 1 else np.minimum(avail, qk)), avail)
        at = row0[None] + bins[..., k]
        idx += [at, at + S * n_bins]
        keep += [served & fifo[None, :, :, k], (qk > 0) & fifo[None, :, :, k]]
    idx = np.concatenate([x.reshape(-1) for x in idx])
    keep = np.concatenate([x.reshape(-1) for x in keep])
    out = np.bincount(idx[keep], minlength=P * 2 * S * n_bins)
    return out.astype(np.uint64).reshape(P, 2, S, n_bins)


def ue_rate_hist(cum_start, cum_end, ue_to_slice, n_slices: int, n_bins: int, bin_bytes: int,
                 cell_profile=None) -> np.ndarray:
    """uint64 [P][S][n_bins]: the samples one ``rs_close_ue_rate_window`` adds (the device twin, bit for bit), from the
    byte counters at the window's start and end.

    cum_start / cum_end: uint64 [B][U] ([B][U][2] with two bearers), ``get_state()["cum_bytes"]``; ue_to_slice [U] or
    [P][U] and cell_profile [B] (None = profile 0): the profiles at close time.  Per UE, c = the sum of its slots and
    d = c_end - c_start, both mod 2^64; bin = min(d // bin_bytes, n_bins - 1), in exact integers."""
    a = np.asarray(cum_start, dtype=np.uint64)
    b = np.asarray(cum_end, dtype=np.uint64)
    B, U = b.shape[:2]
    with np.errstate(over="ignore"):   # uint64 arithmetic wraps, as on the device
        d = b.reshape(B, U, -1).sum(axis=2, dtype=np.uint64) - a.reshape(B, U, -1).sum(axis=2, dtype=np.uint64)
    bins = np.minimum(d // np.uint64(bin_bytes), np.uint64(n_bins - 1)).astype(np.int64)
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    P, S = u2s.shape[0], int(n_slices)
    cp = np.zeros(B, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)
    idx = ((cp[:, None] * S + u2s[cp]) * n_bins + bins).reshape(-1)
    return np.bincount(idx, minlength=P * S * n_bins).astype(np.uint64).reshape(P, S, n_bins)


def ue_upt_hist(queue, cum_start, cum_end, ue_to_slice, n_slices: int, n_bins: int, bin_bytes: int,
                cell_profile=None) -> np.ndarray:
    """uint64 [P][S][n_bins]: the samples one ``rs_close_ue_rate_window`` adds to the throughput-over-active-time
    histograms (``rs_enable_ue_upt_hist``; the device twin, bit for bit).

    queue: the queues the window's TTIs showed, int32 [T][B][U] or [T][B][U][2] (``queue_out``, concatenated over the
    window's run calls); cum_start / cum_end and the profiles as in ``ue_rate_hist``.  A UE is active at a TTI where one
    of its slots shows q > 0; with k > 0 active TTIs it adds bin = min(d // k // bin_bytes, n_bins - 1), d its bytes
    in the window mod 2^64; with k = 0 it adds nothing."""
    a = np.asarray(cum_start, dtype=np.uint64)
    b = np.asarray(cum_end, dtype=np.uint64)
    B, U = b.shape[:2]
    q = np.asarray(queue)
    k = (q.reshape(q.shape[0], B, U, -1) > 0).any(axis=3).sum(axis=0).astype(np.uint64)
    with np.errstate(over="ignore"):   # uint64 arithmetic wraps, as on the device
        d = b.reshape(B, U, -1).sum(axis=2, dtype=np.uint64) - a.reshape(B, U, -1).sum(axis=2, dtype=np.uint64)
    act = k > 0
    bins = np.minimum(d[act] // k[act] // np.uint64(bin_bytes), np.uint64(n_bins - 1)).astype(np.int64)
    u2s = np.atleast_2d(np.asarray(ue_to_slice, dtype=np.int64))
    P, S = u2s.shape[0], int(n_slices)
    cp = np.zeros(B, dtype=np.int64) if cell_profile is None else np.asarray(cell_profile, dtype=np.int64)
    idx = ((cp[:, None] * S + u2s[cp]) * n_bins)[act] + bins
    return np.bincount(idx, minlength=P * S * n_bins).astype(np.uint64).reshape(P, S, n_bins)

"""ctypes binding of the C ABI (include/rs_sched.h -> radiosaber_b200/librs_sched.so).

Host-side mirror of the reference's scheduler plug-in surface for a *batch* of cells: one
:class:`Scheduler` stands for ``n_cells`` independent ``PacketScheduler`` objects of one kind
(ids 1 / 7 / 8 / 9, src/scenarios/single-cell-with-interference.h:94-118) built from the same
slice configuration (:func:`load_slice_config` reads the reference's JSON format,
downlink-transport-scheduler.cpp:55-97), or with :meth:`Scheduler.from_profiles` from several of the same
shape, one per cell.  ``step()`` is one ``Schedule()`` call
(packet-scheduler.cpp:72-90) for every cell.

There is no CPU implementation behind this module: if the CUDA library is missing or no GPU is
present, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RS_SCHED_LIB") or os.path.join(_HERE, "librs_sched.so")
_lib = None

# every symbol include/rs_sched.h declares (tests check the library exports all of them)
ABI_SYMBOLS = (
    "rs_last_error", "rs_abi_version", "rs_create", "rs_destroy", "rs_set_stream", "rs_sync",
    "rs_set_state", "rs_get_state", "rs_reset_state", "rs_step", "rs_run_device", "rs_run_host",
    "rs_synth_cqi", "rs_synth_rand2", "rs_stats_device", "rs_get_stats", "rs_launch_count",
    "rs_smem_bytes", "rs_threads_per_cta", "rs_algorithmic_bytes_per_cell_tti", "rs_test_sort",
    "rs_test_sort_timed", "rs_rand_draws_per_cell_tti", "rs_set_queues",
    "rs_parse_trace_file", "rs_parse_mapping_file", "rs_trace_row", "rs_set_traces",
    "rs_run_traces_device", "rs_run_traces_host",
    "rs_log_create", "rs_log_destroy", "rs_log_set_counters", "rs_log_get_counters", "rs_log_tti", "rs_log_tti_grants",
    "rs_log_stdout", "rs_log_stderr", "rs_log_clear", "rs_log_set_queues", "rs_log_set_app_ids",
    "rs_get_stream", "rs_host_alloc", "rs_host_free", "rs_step_cell", "rs_run_host_async", "rs_run_traces_host_async",
    "rs_wait", "rs_dims", "rs_fixed_shape", "rs_direct_metric",
    "rs_create_profiles", "rs_set_cell_profiles", "rs_n_profiles", "rs_set_grant_list_len", "rs_grant_list_len",
    "rs_enable_buffers", "rs_set_traffic", "rs_get_buffers", "rs_synth_arrivals",
    "rs_buffer_stats_device", "rs_get_buffer_stats", "rs_arrival_spec",
)


class RsError(RuntimeError):
    pass


class _Cfg(C.Structure):
    _fields_ = [
        ("algo", C.c_int32), ("n_slices", C.c_int32), ("n_ues", C.c_int32), ("n_rbs", C.c_int32),
        ("rbg_size", C.c_int32), ("cqi_per_rb", C.c_int32), ("data_to_transmit", C.c_int32),
        ("n_bearers", C.c_int32),
        ("weight", C.c_void_p), ("params", C.c_void_p), ("ue_to_slice", C.c_void_p), ("tbs_row_m1", C.c_void_p),
    ]


class _Out(C.Structure):
    _fields_ = [
        ("rbg_to_ue", C.c_void_p), ("tbs_bits", C.c_void_p), ("mcs", C.c_void_p), ("final_cqi", C.c_void_p),
        ("slice_target", C.c_void_p), ("slice_quota", C.c_void_p), ("nvs_slice", C.c_void_p),
        ("alloc_n", C.c_void_p), ("alloc_ue", C.c_void_p), ("alloc_rbg", C.c_void_p),
    ]


class _CellIo(C.Structure):
    _fields_ = [
        ("avg_rate", C.c_void_p), ("slice_state", C.c_void_p), ("cqi", C.c_void_p), ("rand2", C.c_void_p),
        ("active", C.c_void_p), ("queue_bytes", C.c_void_p), ("hol_delay", C.c_void_p), ("dt", C.c_double),
        ("out", _Out),
    ]


class _Traffic(C.Structure):
    _fields_ = [("arrivals", C.c_void_p), ("now", C.c_void_p), ("arrival_time", C.c_void_p), ("queue_out", C.c_void_p),
                ("hol_out", C.c_void_p)]


def lib():
    """The loaded C ABI library. Raises if it has not been built (``python -c 'import
    __graft_entry__ as g; g.build()'`` or ``make -C radiosaber_b200/csrc``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RsError(f"{LIB_PATH} is missing: build it with `make -C radiosaber_b200/csrc` "
                          "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.rs_last_error.restype = C.c_char_p
        L.rs_abi_version.restype = C.c_int32
        L.rs_create.argtypes = [C.POINTER(_Cfg), C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
        L.rs_create_profiles.argtypes = [C.POINTER(_Cfg), C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                         C.POINTER(C.c_void_p)]
        L.rs_set_cell_profiles.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_n_profiles.argtypes = [C.c_void_p]
        L.rs_n_profiles.restype = C.c_int32
        L.rs_set_grant_list_len.argtypes = [C.c_void_p, C.c_int32]
        L.rs_grant_list_len.argtypes = [C.c_void_p]
        L.rs_grant_list_len.restype = C.c_int32
        L.rs_destroy.argtypes = [C.c_void_p]
        L.rs_destroy.restype = None
        L.rs_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_sync.argtypes = [C.c_void_p]
        L.rs_set_state.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        L.rs_get_state.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        L.rs_reset_state.argtypes = [C.c_void_p]
        L.rs_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.POINTER(_Out)]
        L.rs_run_device.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int64, C.c_void_p, C.POINTER(_Out), C.c_int32]
        L.rs_run_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(_Out), C.c_int32]
        L.rs_synth_cqi.argtypes = [C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p]
        L.rs_synth_rand2.argtypes = [C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p]
        L.rs_stats_device.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_get_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_rand_draws_per_cell_tti.argtypes = [C.c_void_p]
        L.rs_rand_draws_per_cell_tti.restype = C.c_int32
        L.rs_set_queues.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rs_launch_count.argtypes = [C.c_void_p]
        L.rs_launch_count.restype = C.c_int64
        L.rs_smem_bytes.argtypes = [C.c_void_p]
        L.rs_smem_bytes.restype = C.c_int32
        L.rs_threads_per_cta.argtypes = [C.c_void_p]
        L.rs_threads_per_cta.restype = C.c_int32
        L.rs_algorithmic_bytes_per_cell_tti.argtypes = [C.c_void_p]
        L.rs_algorithmic_bytes_per_cell_tti.restype = C.c_int64
        L.rs_test_sort.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        L.rs_test_sort_timed.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                         C.POINTER(C.c_float)]
        L.rs_parse_trace_file.argtypes = [C.c_char_p, C.c_int32, C.c_int32, C.c_void_p]
        L.rs_parse_mapping_file.argtypes = [C.c_char_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
        L.rs_trace_row.argtypes = [C.c_double, C.c_int32]
        L.rs_trace_row.restype = C.c_int32
        L.rs_set_traces.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.rs_run_traces_device.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_void_p, C.POINTER(_Out), C.c_int32]
        L.rs_run_traces_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(_Out), C.c_int32]
        L.rs_log_create.argtypes = [C.POINTER(_Cfg), C.POINTER(C.c_void_p)]
        L.rs_log_destroy.argtypes = [C.c_void_p]
        L.rs_log_destroy.restype = None
        L.rs_log_set_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rs_log_get_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rs_log_set_queues.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rs_log_set_app_ids.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_log_tti.argtypes = [C.c_void_p, C.c_uint64] + [C.c_void_p] * 6
        L.rs_log_tti_grants.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int32] + [C.c_void_p] * 6
        L.rs_log_stdout.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.rs_log_stdout.restype = C.c_char_p
        L.rs_log_stderr.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.rs_log_stderr.restype = C.c_char_p
        L.rs_log_clear.argtypes = [C.c_void_p]
        L.rs_log_clear.restype = None
        L.rs_get_stream.argtypes = [C.c_void_p]
        L.rs_get_stream.restype = C.c_void_p
        L.rs_host_alloc.argtypes = [C.c_size_t, C.c_int32, C.POINTER(C.c_void_p)]
        L.rs_host_free.argtypes = [C.c_void_p]
        L.rs_host_free.restype = None
        L.rs_step_cell.argtypes = [C.c_void_p, C.POINTER(_CellIo)]
        L.rs_run_host_async.argtypes = L.rs_run_host.argtypes + [C.POINTER(C.c_int64)]
        L.rs_run_traces_host_async.argtypes = L.rs_run_traces_host.argtypes + [C.POINTER(C.c_int64)]
        L.rs_wait.argtypes = [C.c_void_p, C.c_int64]
        L.rs_fixed_shape.argtypes = [C.c_void_p]
        L.rs_fixed_shape.restype = C.c_int32
        L.rs_direct_metric.argtypes = [C.c_void_p]
        L.rs_direct_metric.restype = C.c_int32
        L.rs_enable_buffers.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.rs_set_traffic.argtypes = [C.c_void_p, C.POINTER(_Traffic)]
        L.rs_get_buffers.argtypes = [C.c_void_p] + [C.c_void_p] * 4
        L.rs_synth_arrivals.argtypes = [C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
        L.rs_buffer_stats_device.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_get_buffer_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.rs_arrival_spec.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise RsError(f"rs error {rc}: {lib().rs_last_error().decode()}")


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def load_slice_config(path: str):
    """Parse the reference's JSON slice config into (weight[S], params[S][4], ue_to_slice[U]).

    Same expansion as DownlinkTransportScheduler's constructor (downlink-transport-scheduler.cpp:65-88):
    each entry of ``slices`` stands for ``n_slices`` slices with one weight and one
    (alpha, beta, epsilon, psi); ``ues_per_slice[i]`` UEs belong to slice i, UE ids ascending.
    """
    with open(path) as f:
        cfg = json.load(f)
    weight, params = [], []
    for grp in cfg["slices"]:
        for _ in range(int(grp["n_slices"])):
            weight.append(float(grp["weight"]))
            params.append([int(grp["algo_alpha"]), int(grp["algo_beta"]), int(grp["algo_epsilon"]),
                           int(grp["algo_psi"])])
    ue_to_slice = []
    for s, n in enumerate(cfg["ues_per_slice"]):
        ue_to_slice += [s] * int(n)
    if len(cfg["ues_per_slice"]) != len(weight):
        raise ValueError("ues_per_slice does not match the number of slices")
    return (np.asarray(weight, dtype=np.float64), np.asarray(params, dtype=np.int32),
            np.asarray(ue_to_slice, dtype=np.int32))


def arrival_spec(pkt_bytes, pkts_per_tti):
    """(pkt_bytes, pkts_q16) of one slice for :meth:`Scheduler.synth_arrivals` / :func:`workload.synth_arrivals`:
    the rate in 16.16 fixed point, rounded as ``rs_arrival_spec`` rounds it (host only).  ValueError on a value
    the generator does not take."""
    pb, q = C.c_int32(), C.c_int32()
    if lib().rs_arrival_spec(float(pkt_bytes), float(pkts_per_tti), C.byref(pb), C.byref(q)) != 0:
        raise ValueError(lib().rs_last_error().decode())
    return int(pb.value), int(q.value)


def load_traffic_config(path: str, config_path: str):
    """Read a traffic file (the format of ``rs_batch --traffic``) for the slice config at ``config_path``.

    ``{"bearers": 1 | 2, "slices": [...]}``: one entry of ``slices`` per entry of the config's ``slices``, in the same
    order, applying to each of its ``n_slices`` slices: ``{"backlogged": 1}`` (no FIFO) or ``{"pkt_bytes": n,
    "pkts_per_tti": x}``.  Returns (n_bearers, backlogged bool [U][nb], pkt_bytes int32 [S], pkts_q16 int32 [S]);
    ValueError names what is wrong."""
    with open(config_path) as f:
        groups = [int(g["n_slices"]) for g in json.load(f)["slices"]]
    _, _, u2s = load_slice_config(config_path)
    with open(path) as f:
        t = json.load(f)
    where = f"traffic file {path}: "
    if not isinstance(t, dict):
        raise ValueError(where + "not a JSON object")
    nb = t.get("bearers")
    if isinstance(nb, bool) or nb not in (1, 2):
        raise ValueError(where + '"bearers" must be 1 or 2')
    entries = t.get("slices")
    if not isinstance(entries, list):
        raise ValueError(where + '"slices" must be a list')
    if len(entries) != len(groups):
        raise ValueError(where + f'{len(entries)} entries in "slices", the slice config has {len(groups)} slice groups')
    pkt, q16, bl = [], [], []
    num = (int, float)
    for g, e in enumerate(entries):
        at = where + f"slices[{g}]: "
        p = q = 0
        backlogged = isinstance(e, dict) and set(e) == {"backlogged"}
        if backlogged:
            if isinstance(e["backlogged"], bool) or e["backlogged"] != 1:
                raise ValueError(at + '"backlogged" must be 1')
        else:
            if not (isinstance(e, dict) and set(e) == {"pkt_bytes", "pkts_per_tti"}
                    and all(isinstance(e[k], num) and not isinstance(e[k], bool) for k in e)):
                raise ValueError(at + 'expected {"backlogged": 1} or {"pkt_bytes": n, "pkts_per_tti": x}')
            try:
                p, q = arrival_spec(e["pkt_bytes"], e["pkts_per_tti"])
            except ValueError as err:
                raise ValueError(at + str(err)) from None
        pkt += [p] * groups[g]
        q16 += [q] * groups[g]
        bl += [backlogged] * groups[g]
    backlogged = np.repeat(np.asarray(bl, bool)[u2s][:, None], int(nb), axis=1)
    return int(nb), backlogged, np.asarray(pkt, np.int32), np.asarray(q16, np.int32)


class Scheduler:
    """A batch of ``n_cells`` independent cells scheduled on one GPU.

    State (per-bearer EWMA rate and byte counters, per-slice RB offsets / NVS credits) lives in
    device memory between calls, exactly the members the reference keeps in RadioBearer and in
    its scheduler objects (flows/radio-bearer.h:81-85, downlink-transport-scheduler.h:38).
    """

    def __init__(self, algo, weight, params, ue_to_slice, n_cells, n_rbs=512, rbg_size=8, cqi_per_rb=0,
                 data_to_transmit=100000000, tbs_row_m1=None, device=0, n_bearers=1, profiles=None, cell_profile=None):
        """One slice configuration for every cell; or (``profiles``, see :meth:`from_profiles`) several, with
        weight / params / ue_to_slice those of profile 0."""
        self.algo = int(algo)
        self.nb = 2 if int(n_bearers) == 2 else 1   # bearers per UE: per-bearer arrays are [B][U] or [B][U][2]
        self.ue_to_slice = np.ascontiguousarray(ue_to_slice, dtype=np.int32)
        self.U = int(self.ue_to_slice.shape[0])
        self.weight = np.ascontiguousarray(weight, dtype=np.float64)
        self.S = int(self.weight.shape[0])
        self.params = np.ascontiguousarray(params, dtype=np.int32).reshape(self.S, 4)
        self.B = int(n_cells)
        self.R = int(n_rbs)
        self.rbg_size = int(rbg_size)
        self.G = self.R // self.rbg_size
        self.cqi_per_rb = int(cqi_per_rb)
        self.cqi_cols = {0: self.G, 1: self.R, 2: self.G // 2}[self.cqi_per_rb]
        self.device = int(device)
        self._row_m1 = None if tbs_row_m1 is None else np.ascontiguousarray(tbs_row_m1, dtype=np.int32)
        cfg = _Cfg(self.algo, self.S, self.U, self.R, self.rbg_size, self.cqi_per_rb, int(data_to_transmit),
                   int(n_bearers), _ptr(self.weight), _ptr(self.params), _ptr(self.ue_to_slice), _ptr(self._row_m1))
        self._h = C.c_void_p()
        if profiles is None:
            self.n_profiles = 1
            _check(lib().rs_create(C.byref(cfg), self.B, self.device, C.byref(self._h)))
        else:
            # the arrays must outlive the rs_create_profiles call that reads them
            prof = [(np.ascontiguousarray(w, dtype=np.float64), np.ascontiguousarray(p, dtype=np.int32),
                     np.ascontiguousarray(m, dtype=np.int32)) for w, p, m in profiles]
            self.n_profiles = len(prof)
            cfgs = (_Cfg * max(self.n_profiles, 1))()
            for i, (w, p, m) in enumerate(prof):
                cfgs[i] = _Cfg(self.algo, int(w.shape[0]), int(m.shape[0]), self.R, self.rbg_size, self.cqi_per_rb,
                               int(data_to_transmit), int(n_bearers), _ptr(w), _ptr(p), _ptr(m), _ptr(self._row_m1))
            cp = None if cell_profile is None else np.ascontiguousarray(cell_profile, dtype=np.int32).reshape(-1)
            if cp is not None and cp.shape[0] != self.B:
                raise ValueError(f"cell_profile has {cp.shape[0]} entries for {self.B} cells")
            _check(lib().rs_create_profiles(cfgs, len(prof), _ptr(cp), self.B, self.device, C.byref(self._h)))
        # rand() draws per cell-TTI the scheduler consumes: 0 (ids 1/7), 2 (ids 8/9), 300 x largest slice (id 11)
        self.rand_stride = int(lib().rs_rand_draws_per_cell_tti(self._h))

    @classmethod
    def from_config(cls, algo, config_path, n_cells, **kw):
        w, p, u2s = load_slice_config(config_path)
        return cls(algo, w, p, u2s, n_cells, **kw)

    @classmethod
    def from_profiles(cls, algo, profiles, cell_profile, n_cells=None, **kw):
        """Cells with different slice configurations in one batch (rs_create_profiles).  profiles: a list of
        (weight[S], params[S][4], ue_to_slice[U]) as :func:`load_slice_config` returns them, all of the same S and U;
        cell_profile: int [B], the profile of each cell (None only with one profile, then n_cells gives B)."""
        profiles = list(profiles)
        if not profiles:
            raise ValueError("from_profiles needs at least one profile")
        if n_cells is None:
            n_cells = len(cell_profile)
        w, p, m = profiles[0]
        return cls(algo, w, p, m, n_cells, profiles=profiles, cell_profile=cell_profile, **kw)

    def set_cell_profiles(self, cell_profile):
        """A new profile for every cell (rs_set_cell_profiles: waits for the work in flight; state is kept)."""
        cp = np.ascontiguousarray(cell_profile, dtype=np.int32).reshape(-1)
        if cp.shape[0] != self.B:
            raise ValueError(f"cell_profile has {cp.shape[0]} entries for {self.B} cells")
        _check(lib().rs_set_cell_profiles(self._h, _ptr(cp)))

    @property
    def grant_list_len(self):
        """Id 10: entries per cell of the alloc_ue / alloc_rbg outputs (0 for other ids)."""
        return int(lib().rs_grant_list_len(self._h))

    def set_grant_list_len(self, n):
        """Id 10: list n grants per cell, 2G (the default) .. S*G (every grant; rs_set_grant_list_len).  The schedule
        never depends on it: alloc_n counts every grant, the list holds the first n."""
        _check(lib().rs_set_grant_list_len(self._h, int(n)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().rs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state -------------------------------------------------------------------------------
    def set_state(self, avg_rate=None, tx_bytes=None, slice_offset=None, nvs_ewma=None, cum_bytes=None,
                  cum_rbs=None):
        B, U, S = self.B, self.U, self.S
        BU = (B, U) if self.nb == 1 else (B, U, 2)

        def arr(v, dt, shape):
            return None if v is None else np.ascontiguousarray(np.asarray(v).reshape(shape), dtype=dt)

        a = arr(avg_rate, np.float64, BU); t = arr(tx_bytes, np.int32, BU)
        cb = arr(cum_bytes, np.uint64, BU); cr = arr(cum_rbs, np.uint64, BU)
        so = arr(slice_offset, np.float64, (B, S)); ne = arr(nvs_ewma, np.float64, (B, S))
        _check(lib().rs_set_state(self._h, _ptr(a), _ptr(t), _ptr(cb), _ptr(cr), _ptr(so), _ptr(ne)))

    def get_state(self):
        B, U, S = self.B, self.U, self.S
        BU = (B, U) if self.nb == 1 else (B, U, 2)
        st = {"avg_rate": np.empty(BU, np.float64), "tx_bytes": np.empty(BU, np.int32),
              "cum_bytes": np.empty(BU, np.uint64), "cum_rbs": np.empty(BU, np.uint64),
              "slice_offset": np.empty((B, S), np.float64), "nvs_ewma": np.empty((B, S), np.float64)}
        _check(lib().rs_get_state(self._h, _ptr(st["avg_rate"]), _ptr(st["tx_bytes"]), _ptr(st["cum_bytes"]),
                                  _ptr(st["cum_rbs"]), _ptr(st["slice_offset"]), _ptr(st["nvs_ewma"])))
        return st

    def reset_state(self):
        _check(lib().rs_reset_state(self._h))

    # ---- host-buffer path --------------------------------------------------------------------
    def _host_outputs(self, T, want_aux):
        B, U, S, G = self.B, self.U, self.S, self.G
        lead = (T, B) if T is not None else (B,)
        out = {"rbg_to_ue": np.empty(lead + (G,), np.int16), "tbs_bits": np.empty(lead + (U,), np.int32),
               "mcs": np.empty(lead + (U,), np.uint8)}
        if want_aux:
            out["final_cqi"] = np.empty(lead + (U,), np.uint8)
            if self.algo == 10:
                out["alloc_n"] = np.empty(lead, np.int32)
                out["alloc_ue"] = np.empty(lead + (self.grant_list_len,), np.int16)
                out["alloc_rbg"] = np.empty(lead + (self.grant_list_len,), np.int16)
            if self.algo in (8, 9, 10, 101, 103):
                out["slice_target"] = np.empty(lead + (S,), np.int32)
                out["slice_quota"] = np.empty(lead + (S,), np.int32)
            if self.algo in (7, 11):
                out["nvs_slice"] = np.empty(lead, np.int32)
        o = _Out(*[_ptr(out.get(k)) for k in ("rbg_to_ue", "tbs_bits", "mcs", "final_cqi", "slice_target",
                                                "slice_quota", "nvs_slice", "alloc_n", "alloc_ue", "alloc_rbg")])
        return out, o

    def _draws(self, rand2, lead):
        """rand() draws as int32 lead + (rand_stride,); a wider array (recorded draws padded to the largest
        TTI) is cut or zero-padded to the stride; ids without draws get a dummy."""
        n = max(self.rand_stride, 2)
        if rand2 is None:
            return np.zeros(lead + (n,), dtype=np.int32)
        r = np.asarray(rand2, dtype=np.int32)
        r = r.reshape(lead + (-1,))
        if r.shape[-1] < n:
            r = np.concatenate([r, np.zeros(lead + (n - r.shape[-1],), dtype=np.int32)], axis=-1)
        return np.ascontiguousarray(r[..., :n])

    def _queues(self, queue, hol, lead):
        """Hand the next run call its queue state (rs_set_queues); returns the arrays to keep alive."""
        if queue is None:
            return None
        per_ue = (self.U,) if self.nb == 1 else (self.U, 2)
        q = np.ascontiguousarray(queue, dtype=np.int32).reshape(lead + per_ue)
        h = None if hol is None else np.ascontiguousarray(hol, dtype=np.float64).reshape(lead + per_ue)
        _check(lib().rs_set_queues(self._h, _ptr(q), _ptr(h)))
        return q, h

    # ---- per-bearer buffers on the device (closed-loop queues, rs_enable_buffers) -------------------
    def enable_buffers(self, max_records, backlogged=None):
        """Keep a byte FIFO of at most max_records records per bearer on the device (0 = off); backlogged: bool
        [B][U] ([B][U][2] with two bearers) of bearers without a FIFO (the infinite buffer).  Empties every FIFO."""
        bl = None if backlogged is None else np.ascontiguousarray(np.asarray(backlogged).reshape(self._per_bearer((self.B,))),
                                                                  dtype=np.uint8)
        _check(lib().rs_enable_buffers(self._h, int(max_records), _ptr(bl)))

    def get_buffers(self):
        """{queued int64, n_records int32, head_time float64, dropped uint64}, each [B][U] ([B][U][2])."""
        shape = self._per_bearer((self.B,))
        st = {"queued": np.empty(shape, np.int64), "n_records": np.empty(shape, np.int32),
              "head_time": np.empty(shape, np.float64), "dropped": np.empty(shape, np.uint64)}
        _check(lib().rs_get_buffers(self._h, *[_ptr(st[k]) for k in ("queued", "n_records", "head_time", "dropped")]))
        return st

    def get_buffer_stats(self):
        """uint64 [3][S]: per slice, the bytes queued, the bytes dropped and the records held over the bearers with a
        FIFO; [P][3][S] with P > 1 slice profiles, row p over the cells of profile p (rs_get_buffer_stats)."""
        st = np.empty((self.n_profiles, 3, self.S), dtype=np.uint64)
        _check(lib().rs_get_buffer_stats(self._h, _ptr(st)))
        return st[0] if self.n_profiles == 1 else st

    def buffer_stats_device(self, d_stats):
        """rs_buffer_stats_device into a DEVICE buffer of n_profiles * 3 * S uint64."""
        _check(lib().rs_buffer_stats_device(self._h, C.c_void_p(d_stats)))

    def synth_arrivals(self, seed, cell0, tti0, n_ttis, pkt_bytes, pkts_q16, d_out):
        """rs_synth_arrivals: int32 [n_ttis][B][U][nb] into device memory; pkt_bytes / pkts_q16: int [P][S] (packet
        size, packets per TTI in 16.16 fixed point) per slice of each profile.  Twin of workload.synth_arrivals."""
        pb = np.ascontiguousarray(np.asarray(pkt_bytes).reshape(self.n_profiles, self.S), dtype=np.int32)
        pq = np.ascontiguousarray(np.asarray(pkts_q16).reshape(self.n_profiles, self.S), dtype=np.int32)
        _check(lib().rs_synth_arrivals(self._h, int(seed), int(cell0), int(tti0), int(n_ttis), _ptr(pb), _ptr(pq),
                                       C.c_void_p(d_out)))

    def _per_bearer(self, lead):
        return lead + ((self.U,) if self.nb == 1 else (self.U, 2))

    def _traffic(self, arrivals, now, arrival_time, T, out):
        """Hand the next HOST run call of T TTIs its traffic (rs_set_traffic); the queue sizes and delays the TTIs show go
        to out["queue_out"] / out["hol_out"].  Returns the arrays to keep alive."""
        if arrivals is None:
            return None
        lead = (T, self.B) if T is not None else (self.B,)
        n = 1 if T is None else T
        a = np.ascontiguousarray(arrivals, dtype=np.int32).reshape(self._per_bearer(lead))
        nw = np.ascontiguousarray(np.asarray(now, dtype=np.float64).reshape(n))
        at = nw if arrival_time is None else np.ascontiguousarray(np.asarray(arrival_time, dtype=np.float64).reshape(n))
        out["queue_out"] = np.empty(a.shape, np.int32)
        out["hol_out"] = np.empty(a.shape, np.float64)
        tr = _Traffic(_ptr(a), _ptr(nw), _ptr(at), _ptr(out["queue_out"]), _ptr(out["hol_out"]))
        _check(lib().rs_set_traffic(self._h, C.byref(tr)))
        return a, nw, at

    def _device_traffic(self, n_ttis, d_arrivals, now, arrival_time, d_queue_out, d_hol_out):
        """Hand the next DEVICE run call its traffic: arrivals / outputs are device pointers, now / arrival_time host
        arrays [T].  Returns the arrays to keep alive."""
        if not d_arrivals:
            return None
        nw = np.ascontiguousarray(np.asarray(now, dtype=np.float64).reshape(-1)[:n_ttis])
        at = nw if arrival_time is None else np.ascontiguousarray(np.asarray(arrival_time, dtype=np.float64).reshape(-1)[:n_ttis])
        tr = _Traffic(C.c_void_p(d_arrivals), _ptr(nw), _ptr(at), C.c_void_p(d_queue_out or None), C.c_void_p(d_hol_out or None))
        _check(lib().rs_set_traffic(self._h, C.byref(tr)))
        return nw, at

    def step(self, cqi, rand2=None, dt=0.001, active=None, want_aux=False, queue=None, hol=None, arrivals=None, now=None,
             arrival_time=None):
        """One TTI for every cell. cqi: uint8 [B][U][G] (or [B][U][R]); rand2: int32 [B][2]; queue / hol: the
        bearers' dataToTransmit (int32 [B][U]) and head-of-line delays (float64 [B][U]), see rs_set_queues.  A buffered
        handle takes arrivals (int32 [B][U]), now and arrival_time (default now) instead, and returns the queue sizes and
        delays the TTI showed as out["queue_out"] / out["hol_out"] (rs_set_traffic)."""
        B, U = self.B, self.U
        keep = self._queues(queue, hol, (B,))
        cqi = np.ascontiguousarray(cqi, dtype=np.uint8)
        assert cqi.size == B * U * self.cqi_cols, cqi.shape
        rand2 = self._draws(rand2, (B,))
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(B, U)
        out, o = self._host_outputs(None, want_aux)
        keep_tr = self._traffic(arrivals, now, arrival_time, None, out)
        _check(lib().rs_step(self._h, _ptr(cqi), _ptr(rand2), _ptr(act), float(dt), C.byref(o)))
        return out

    def step_cell(self, cqi, rand2=None, dt=0.001, active=None, queue=None, hol=None, avg_rate=None,
                  slice_state=None):
        """rs_step_cell: one TTI with the caller's state (avg_rate [B][U], slice_state [B][S], both updated in
        place when given) travelling with the inputs -- one copy up, one launch, one copy down."""
        B, U = self.B, self.U
        cqi = np.ascontiguousarray(cqi, dtype=np.uint8)
        assert cqi.size == B * U * self.cqi_cols, cqi.shape
        rand2 = self._draws(rand2, (B,))
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(B, U)
        q = None if queue is None else np.ascontiguousarray(queue, dtype=np.int32).reshape(B, U)
        h = None if hol is None else np.ascontiguousarray(hol, dtype=np.float64).reshape(B, U)
        for st, shape in ((avg_rate, (B, U)), (slice_state, (B, self.S))):
            assert st is None or (st.dtype == np.float64 and st.flags.c_contiguous and st.shape == shape)
        out, o = self._host_outputs(None, True)
        io = _CellIo(_ptr(avg_rate), _ptr(slice_state), _ptr(cqi), _ptr(rand2), _ptr(act), _ptr(q), _ptr(h), float(dt), o)
        _check(lib().rs_step_cell(self._h, C.byref(io)))
        return out

    def run_host_async(self, cqi, rand2, dt, out, o, ttis_per_launch=0, cqi_refresh=1, traffic=None):
        """rs_run_host_async on caller-owned arrays (kept alive and untouched until wait(ticket)); out / o come from
        _host_outputs().  traffic: (arrivals, now, arrival_time) of a buffered handle, whose arrays the caller keeps alive
        as well (the shown queues and delays land in out["queue_out"] / out["hol_out"]).  Returns the ticket."""
        T = int(dt.shape[0])
        if traffic is not None:
            a, nw, at = traffic
            out["queue_out"] = np.empty(a.shape, np.int32)
            out["hol_out"] = np.empty(a.shape, np.float64)
            tr = _Traffic(_ptr(a), _ptr(nw), _ptr(at), _ptr(out["queue_out"]), _ptr(out["hol_out"]))
            _check(lib().rs_set_traffic(self._h, C.byref(tr)))
        ticket = C.c_int64(-1)
        _check(lib().rs_run_host_async(self._h, T, _ptr(cqi), int(cqi_refresh), _ptr(rand2), None, _ptr(dt),
                                       C.byref(o), int(ttis_per_launch), C.byref(ticket)))
        return int(ticket.value)

    def wait(self, ticket):
        _check(lib().rs_wait(self._h, int(ticket)))

    def run_host(self, cqi, rand2, dt, active=None, want_aux=False, ttis_per_launch=0, cqi_refresh=1, queue=None,
                 hol=None, arrivals=None, now=None, arrival_time=None):
        """T TTIs with host arrays [T][B][...] (cqi: one slab per cqi_refresh TTIs); copies overlap
        the kernels.  arrivals [T][B][U] / now [T] / arrival_time [T]: as step() for a buffered handle."""
        B, U = self.B, self.U
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        T = int(dt.shape[0])
        cqi = np.ascontiguousarray(cqi, dtype=np.uint8)
        assert cqi.size == -(-T // cqi_refresh) * B * U * self.cqi_cols, cqi.shape
        rand2 = None if rand2 is None else self._draws(rand2, (T, B))
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(T, B, U)
        out, o = self._host_outputs(T, want_aux)
        keep = self._queues(queue, hol, (T, B))
        keep_tr = self._traffic(arrivals, now, arrival_time, T, out)
        _check(lib().rs_run_host(self._h, T, _ptr(cqi), int(cqi_refresh), _ptr(rand2), _ptr(act), _ptr(dt),
                                 C.byref(o), int(ttis_per_launch)))
        return out

    # ---- device-resident path (raw device pointers, e.g. torch tensors' data_ptr()) -----------
    def _device_queues(self, d_queue, d_hol):
        """Hand the next run call DEVICE queue state ([T][B][U] or [T][B][U][2] int32 / float64, rs_set_queues)."""
        if d_queue or d_hol:
            _check(lib().rs_set_queues(self._h, C.c_void_p(d_queue or None), C.c_void_p(d_hol or None)))

    def run_device(self, n_ttis, d_cqi, cqi_tti_stride, d_rand2, dt, d_out=None, d_active=0,
                   active_tti_stride=0, ttis_per_launch=0, cqi_refresh=1, d_queue=0, d_hol=0, d_arrivals=0, now=None,
                   arrival_time=None, d_queue_out=0, d_hol_out=0):
        """d_arrivals / d_queue_out / d_hol_out: device pointers of a buffered handle's traffic ([T][B][U][nb]); now /
        arrival_time host arrays [T] (rs_set_traffic)."""
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        assert dt.shape[0] >= n_ttis
        self._device_queues(d_queue, d_hol)
        keep_tr = self._device_traffic(n_ttis, d_arrivals, now, arrival_time, d_queue_out, d_hol_out)
        o = _Out(*[(d_out or {}).get(k) for k in ("rbg_to_ue", "tbs_bits", "mcs", "final_cqi", "slice_target",
                                                    "slice_quota", "nvs_slice", "alloc_n", "alloc_ue", "alloc_rbg")])
        _check(lib().rs_run_device(self._h, int(n_ttis), C.c_void_p(d_cqi), int(cqi_tti_stride), int(cqi_refresh),
                                   C.c_void_p(d_rand2 or None), C.c_void_p(d_active or None),
                                   int(active_tti_stride), _ptr(dt), C.byref(o), int(ttis_per_launch)))

    # ---- trace-driven CQI (enb-mac-entity.cc:42-56, 160-193) ----------------------------------
    def set_traces(self, traces, ue_trace):
        """traces: uint8 [n_traces][n_rows][n_rbs] (see :func:`load_trace_dir`); ue_trace: int32 [B][U],
        the trace every UE of every cell replays."""
        traces = np.ascontiguousarray(traces, dtype=np.uint8)
        assert traces.ndim == 3 and traces.shape[2] == self.R, traces.shape
        ue_trace = np.ascontiguousarray(np.broadcast_to(np.asarray(ue_trace, dtype=np.int32), (self.B, self.U)))
        _check(lib().rs_set_traces(self._h, _ptr(traces), traces.shape[0], traces.shape[1], _ptr(ue_trace)))
        self.trace_rows = int(traces.shape[1])

    def run_traces_host(self, trace_row, rand2, dt, active=None, want_aux=False, ttis_per_launch=0, queue=None,
                        hol=None, arrivals=None, now=None, arrival_time=None):
        """T TTIs with the CQI replayed from the loaded traces; trace_row: int32 [T] (-1 = no report yet); queue / hol
        and arrivals / now / arrival_time as run_host."""
        B, U = self.B, self.U
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        T = int(dt.shape[0])
        trace_row = np.ascontiguousarray(trace_row, dtype=np.int32)
        assert trace_row.shape == (T,)
        rand2 = None if rand2 is None else self._draws(rand2, (T, B))
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(T, B, U)
        out, o = self._host_outputs(T, want_aux)
        keep = self._queues(queue, hol, (T, B))
        keep_tr = self._traffic(arrivals, now, arrival_time, T, out)
        _check(lib().rs_run_traces_host(self._h, T, _ptr(trace_row), _ptr(rand2), _ptr(act), _ptr(dt), C.byref(o),
                                        int(ttis_per_launch)))
        return out

    def run_traces_device(self, n_ttis, trace_row, d_rand2, dt, d_out=None, d_active=0, active_tti_stride=0,
                          ttis_per_launch=0, d_queue=0, d_hol=0, d_arrivals=0, now=None, arrival_time=None, d_queue_out=0,
                          d_hol_out=0):
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        trace_row = np.ascontiguousarray(trace_row, dtype=np.int32)
        assert dt.shape[0] >= n_ttis and trace_row.shape[0] >= n_ttis
        self._device_queues(d_queue, d_hol)
        keep_tr = self._device_traffic(n_ttis, d_arrivals, now, arrival_time, d_queue_out, d_hol_out)
        o = _Out(*[(d_out or {}).get(k) for k in ("rbg_to_ue", "tbs_bits", "mcs", "final_cqi", "slice_target",
                                                    "slice_quota", "nvs_slice", "alloc_n", "alloc_ue", "alloc_rbg")])
        _check(lib().rs_run_traces_device(self._h, int(n_ttis), _ptr(trace_row), C.c_void_p(d_rand2 or None),
                                          C.c_void_p(d_active or None), int(active_tti_stride), _ptr(dt),
                                          C.byref(o), int(ttis_per_launch)))

    def synth_cqi(self, seed, cell0, epoch0, n_slabs, d_out):
        """n_slabs CQI slabs [B][U][row] for epochs epoch0.. (epoch = tti // refresh) into device memory."""
        _check(lib().rs_synth_cqi(self._h, int(seed), int(cell0), int(epoch0), int(n_slabs), C.c_void_p(d_out)))

    def synth_rand2(self, seed, cell0, tti0, n_ttis, d_out):
        _check(lib().rs_synth_rand2(self._h, int(seed), int(cell0), int(tti0), int(n_ttis), C.c_void_p(d_out)))

    def set_stream(self, cuda_stream):
        _check(lib().rs_set_stream(self._h, C.c_void_p(cuda_stream or None)))

    def sync(self):
        _check(lib().rs_sync(self._h))

    def stats_device(self, d_stats):
        """rs_stats_device into a DEVICE buffer of n_profiles * 4 * S uint64 ([P][4][S], [4][S] with one profile)."""
        _check(lib().rs_stats_device(self._h, C.c_void_p(d_stats)))

    def get_stats(self):
        """uint64 [4][S]: sum bytes, sum RBs, sum q, sum q^2 (q = UE cumulative bytes >> 10); [P][4][S] with P > 1
        slice profiles, row p over the cells of profile p."""
        st = np.empty((self.n_profiles, 4, self.S), dtype=np.uint64)
        _check(lib().rs_get_stats(self._h, _ptr(st)))
        return st[0] if self.n_profiles == 1 else st

    @property
    def launch_count(self):
        return int(lib().rs_launch_count(self._h))

    @property
    def smem_bytes(self):
        return int(lib().rs_smem_bytes(self._h))

    @property
    def algorithmic_bytes_per_cell_tti(self):
        return int(lib().rs_algorithmic_bytes_per_cell_tti(self._h))


class LogWriter:
    """The reference's per-TTI stdout / stderr text for ONE cell, regenerated from batch results
    (downlink-transport-scheduler.cpp:192-199, 523-527, 631-649; host only).  With slice profiles, pass the
    ue_to_slice of the logged cell's own profile."""

    def __init__(self, algo, ue_to_slice, n_slices, n_rbs=512, rbg_size=8, cqi_per_rb=0,
                 data_to_transmit=100000000, n_bearers=1, app_ids=None):
        self._u2s = np.ascontiguousarray(ue_to_slice, dtype=np.int32)
        self.U, self.S, self.G = int(self._u2s.shape[0]), int(n_slices), int(n_rbs) // int(rbg_size)
        self.nb = 2 if int(n_bearers) == 2 else 1   # per-bearer arrays (queue, hol, counters, app ids) are [U] or [U][2]
        cfg = _Cfg(int(algo), self.S, self.U, int(n_rbs), int(rbg_size), int(cqi_per_rb), int(data_to_transmit), int(n_bearers),
                   None, None, _ptr(self._u2s), None)
        self._h = C.c_void_p()
        _check(lib().rs_log_create(C.byref(cfg), C.byref(self._h)))
        if app_ids is not None:
            a = np.ascontiguousarray(app_ids, dtype=np.int32)
            assert a.size == self.U * self.nb
            _check(lib().rs_log_set_app_ids(self._h, _ptr(a)))

    def tti(self, timestamp, cqi, rbg_to_ue, tbs_bits, final_cqi=None, slice_target=None, slice_quota=None,
            queue=None, hol=None):
        if queue is not None or hol is not None:
            q = None if queue is None else np.ascontiguousarray(queue, dtype=np.int32)
            h = None if hol is None else np.ascontiguousarray(hol, dtype=np.float64)
            _check(lib().rs_log_set_queues(self._h, _ptr(q), _ptr(h)))
        a = [np.ascontiguousarray(cqi, dtype=np.uint8), np.ascontiguousarray(rbg_to_ue, dtype=np.int16),
             np.ascontiguousarray(tbs_bits, dtype=np.int32),
             None if final_cqi is None else np.ascontiguousarray(final_cqi, dtype=np.uint8),
             None if slice_target is None else np.ascontiguousarray(slice_target, dtype=np.int32),
             None if slice_quota is None else np.ascontiguousarray(slice_quota, dtype=np.int32)]
        _check(lib().rs_log_tti(self._h, int(timestamp), *[_ptr(x) for x in a]))

    def tti_grants(self, timestamp, cqi, n_grants, grant_ue, grant_rbg, tbs_bits, final_cqi, slice_target, slice_quota,
                   queue=None, hol=None):
        """Id 10: one TTI from the grant list (rs_outputs.alloc_*) instead of the single-valued RBG->UE map.  grant_ue /
        grant_rbg hold n_grants entries: a handle's list of rs_grant_list_len >= alloc_n (S*G always is)."""
        if queue is not None or hol is not None:
            q = None if queue is None else np.ascontiguousarray(queue, dtype=np.int32)
            h = None if hol is None else np.ascontiguousarray(hol, dtype=np.float64)
            _check(lib().rs_log_set_queues(self._h, _ptr(q), _ptr(h)))
        a = [np.ascontiguousarray(grant_ue, dtype=np.int16), np.ascontiguousarray(grant_rbg, dtype=np.int16),
             np.ascontiguousarray(tbs_bits, dtype=np.int32), np.ascontiguousarray(final_cqi, dtype=np.uint8),
             np.ascontiguousarray(slice_target, dtype=np.int32), np.ascontiguousarray(slice_quota, dtype=np.int32)]
        c = np.ascontiguousarray(cqi, dtype=np.uint8)
        assert a[0].size >= int(n_grants) and a[1].size >= int(n_grants)   # every grant of the TTI
        _check(lib().rs_log_tti_grants(self._h, int(timestamp), _ptr(c), int(n_grants), *[_ptr(x) for x in a]))

    def set_counters(self, cum_bytes=None, cum_rbs=None):
        cb = None if cum_bytes is None else np.ascontiguousarray(cum_bytes, dtype=np.uint64)
        cr = None if cum_rbs is None else np.ascontiguousarray(cum_rbs, dtype=np.uint64)
        _check(lib().rs_log_set_counters(self._h, _ptr(cb), _ptr(cr)))

    def counters(self):
        shape = (self.U,) if self.nb == 1 else (self.U, 2)
        cb, cr = np.empty(shape, np.uint64), np.empty(shape, np.uint64)
        _check(lib().rs_log_get_counters(self._h, _ptr(cb), _ptr(cr)))
        return cb, cr

    @property
    def stdout(self) -> str:
        return lib().rs_log_stdout(self._h, None).decode()

    @property
    def stderr(self) -> str:
        return lib().rs_log_stderr(self._h, None).decode()

    def clear(self):
        lib().rs_log_clear(self._h)

    def close(self):
        if getattr(self, "_h", None):
            lib().rs_log_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pack_cqi(cqi: np.ndarray) -> np.ndarray:
    """u8 [..., G] (values 1..15) -> the 4-bit layout (cqi_per_rb = 2): [..., G/2], even RBG in the low nibble."""
    cqi = np.asarray(cqi, dtype=np.uint8)
    return np.ascontiguousarray(cqi[..., 0::2] | (cqi[..., 1::2] << 4))


# ---- trace files (host only; no GPU needed) ---------------------------------------------------------
TRACE_ROWS = 475      # MAX_TTI_TRACE, enb-mac-entity.cc:40
CQI_INTERVAL = 40     # enb-mac-entity.cc:38 and the UEs' reporting interval (single-cell-with-interference.h:276-278)


def parse_trace_file(path, n_rows=TRACE_ROWS, n_rbs=512) -> np.ndarray:
    """uint8 [n_rows][n_rbs]: one ue<id>.log as the reference reads it (enb-mac-entity.cc:169-187)."""
    out = np.empty((n_rows, n_rbs), dtype=np.uint8)
    _check(lib().rs_parse_trace_file(os.fsencode(path), n_rows, n_rbs, _ptr(out)))
    return out


def parse_mapping_file(path) -> np.ndarray:
    """int32 [n]: the trace ids of a mapping.config in file order (enb-mac-entity.cc:48-55)."""
    n = C.c_int32(0)
    _check(lib().rs_parse_mapping_file(os.fsencode(path), None, 0, C.byref(n)))
    out = np.empty(n.value, dtype=np.int32)
    _check(lib().rs_parse_mapping_file(os.fsencode(path), _ptr(out), n.value, C.byref(n)))
    return out


def load_trace_dir(trace_dir, trace_ids=None, n_rows=TRACE_ROWS, n_rbs=512):
    """(traces uint8 [n][n_rows][n_rbs], ids int32 [n]) for the ue<id>.log files of a cqi-traces directory."""
    if trace_ids is None:
        trace_ids = sorted(int(f[2:-4]) for f in os.listdir(trace_dir) if f.startswith("ue") and f.endswith(".log"))
    ids = np.asarray(list(trace_ids), dtype=np.int32)
    traces = np.stack([parse_trace_file(os.path.join(trace_dir, f"ue{int(i)}.log"), n_rows, n_rbs) for i in ids])
    return traces, ids


def trace_row(now_seconds, n_rows=TRACE_ROWS) -> int:
    """(int)(Now*1000/40) % n_rows, enb-mac-entity.cc:189-191."""
    return int(lib().rs_trace_row(float(now_seconds), int(n_rows)))


def trace_rows_for_run(now, first_report_tti=0, interval=CQI_INTERVAL, n_rows=TRACE_ROWS) -> np.ndarray:
    """int32 [T]: the trace line in force at every TTI of a run whose TTI t happens at now[t] when the
    UEs report at TTIs first_report_tti, first_report_tti + interval, ... (-1 before the first report)."""
    now = np.asarray(now, dtype=np.float64)
    rows = np.full(now.shape[0], -1, dtype=np.int32)
    for t in range(now.shape[0]):
        if t >= first_report_tti:
            last = first_report_tti + (t - first_report_tti) // interval * interval
            rows[t] = trace_row(now[last], n_rows)
    return rows


def test_sort(keys, depth_limit=-1, device=0) -> np.ndarray:
    """Device std::sort order (key descending) of each row of uint8 keys[n_arrays][n]."""
    keys = np.ascontiguousarray(keys, dtype=np.uint8)
    if keys.ndim == 1:
        keys = keys[None]
    perm = np.empty(keys.shape, dtype=np.int32)
    _check(lib().rs_test_sort(int(device), _ptr(keys), keys.shape[0], keys.shape[1], int(depth_limit), _ptr(perm)))
    return perm


def test_sort_timed(keys, reps=20, depth_limit=-1, device=0):
    """(perm, ms per launch) of the device sort over all rows of keys (development aid)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint8)
    perm = np.empty(keys.shape, dtype=np.int32)
    ms = C.c_float(0)
    _check(lib().rs_test_sort_timed(int(device), _ptr(keys), keys.shape[0], keys.shape[1], int(depth_limit),
                                    _ptr(perm), int(reps), C.byref(ms)))
    return perm, float(ms.value)


def jain_index(stats: np.ndarray, n_ues_per_slice: np.ndarray) -> np.ndarray:
    """Per-slice Jain fairness (sum q)^2 / (n * sum q^2) from rs_get_stats() totals."""
    sq = stats[2].astype(np.float64)
    sqq = stats[3].astype(np.float64)
    n = np.asarray(n_ues_per_slice, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(sqq > 0, sq * sq / (n * sqq), 0.0)

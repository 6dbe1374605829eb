"""ctypes binding for oracle/librs_oracle.so (the CPU restatement).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package
(radiosaber_b200/) never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "librs_oracle.so")
_lib = None


class _Cfg(C.Structure):
    _fields_ = [
        ("algo", C.c_int32), ("n_slices", C.c_int32), ("n_ues", C.c_int32), ("n_rbs", C.c_int32),
        ("rbg_size", C.c_int32), ("cqi_per_rb", C.c_int32), ("data_to_transmit", C.c_int32),
        ("dead_work", C.c_int32), ("n_bearers", C.c_int32), ("reserved", C.c_int32),
        ("weight", C.c_void_p), ("params", C.c_void_p), ("ue_to_slice", C.c_void_p), ("tbs_row_m1", C.c_void_p),
    ]


class _Io(C.Structure):
    _fields_ = [
        ("avg_rate", C.c_void_p), ("tx_bytes", C.c_void_p), ("cum_bytes", C.c_void_p), ("cum_rbs", C.c_void_p),
        ("slice_offset", C.c_void_p), ("nvs_ewma", C.c_void_p),
        ("cqi", C.c_void_p), ("active", C.c_void_p), ("rand2", C.c_void_p), ("dt", C.c_double),
        ("rbg_to_ue", C.c_void_p), ("tbs_bits", C.c_void_p), ("mcs", C.c_void_p), ("final_cqi", C.c_void_p),
        ("slice_target", C.c_void_p), ("slice_quota", C.c_void_p), ("nvs_slice", C.c_void_p),
        ("alloc_n", C.c_void_p), ("alloc_ue", C.c_void_p), ("alloc_rbg", C.c_void_p),
        ("rand_stride", C.c_int32),
        ("queue_bytes", C.c_void_p), ("hol_delay", C.c_void_p), ("alloc_len", C.c_int32),
    ]


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "rs_oracle.cpp")
    stale = (not os.path.exists(_LIB_PATH)) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src)
    if force or stale:
        subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.rso_step.restype = C.c_int
        _lib.rso_step.argtypes = [C.POINTER(_Cfg), C.c_int32, C.POINTER(_Io), C.c_int32]
        _lib.rso_eesm_effective_sinr.restype = C.c_double
        _lib.rso_eesm_effective_sinr.argtypes = [C.c_void_p, C.c_int32]
        _lib.rso_cqi_from_sinr.restype = C.c_int32
        _lib.rso_cqi_from_sinr.argtypes = [C.c_double]
        _lib.rso_sinr_from_cqi.restype = C.c_double
        _lib.rso_sinr_from_cqi.argtypes = [C.c_int32]
        _lib.rso_mcs_from_cqi.restype = C.c_int32
        _lib.rso_mcs_from_cqi.argtypes = [C.c_int32]
        _lib.rso_tbs_from_mcs.restype = C.c_int32
        _lib.rso_tbs_from_mcs.argtypes = [C.c_int32, C.c_int32, C.c_void_p]
        _lib.rso_efficiency_from_cqi.restype = C.c_double
        _lib.rso_efficiency_from_cqi.argtypes = [C.c_int32]
        _lib.rso_std_sort_desc.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        _lib.rso_introsort_emul_desc.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class OracleScheduler:
    """Batch of independent cells stepped by the CPU restatement.

    State arrays live in numpy and are updated in place, mirroring what the
    reference keeps per bearer / per scheduler object.
    """

    def __init__(self, algo, weight, params, ue_to_slice, n_cells, n_rbs=512, rbg_size=8, cqi_per_rb=0,
                 data_to_transmit=100000000, dead_work=0, tbs_row_m1=None, n_threads=1, n_bearers=1,
                 grant_list_len=None):
        """grant_list_len: id 10, entries per cell of the alloc_ue / alloc_rbg outputs (default 2G, S*G lists every
        grant); alloc_n counts every grant whatever the length."""
        self.algo = int(algo)
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
        self.n_threads = int(n_threads)
        self._row_m1 = None if tbs_row_m1 is None else np.ascontiguousarray(tbs_row_m1, dtype=np.int32)
        self.nb = 2 if int(n_bearers) == 2 else 1
        self.grant_list_len = 2 * self.G if grant_list_len is None else int(grant_list_len)
        self._cfg = _Cfg(self.algo, self.S, self.U, self.R, self.rbg_size, self.cqi_per_rb,
                         int(data_to_transmit), int(dead_work), int(n_bearers), 0,
                         _ptr(self.weight), _ptr(self.params), _ptr(self.ue_to_slice), _ptr(self._row_m1))
        B, U, S = self.B, self.U, self.S
        BU = (B, U) if self.nb == 1 else (B, U, 2)   # per-bearer state
        self.avg_rate = np.full(BU, 100000.0, dtype=np.float64)   # radio-bearer.cpp:54
        self.tx_bytes = np.zeros(BU, dtype=np.int32)
        self.cum_bytes = np.zeros(BU, dtype=np.uint64)
        self.cum_rbs = np.zeros(BU, dtype=np.uint64)
        self.slice_offset = np.zeros((B, S), dtype=np.float64)
        self.nvs_ewma = np.zeros((B, S), dtype=np.float64)

    def set_state(self, avg_rate=None, tx_bytes=None, slice_offset=None, nvs_ewma=None, cum_bytes=None,
                  cum_rbs=None):
        for name, val in (("avg_rate", avg_rate), ("tx_bytes", tx_bytes), ("slice_offset", slice_offset),
                          ("nvs_ewma", nvs_ewma), ("cum_bytes", cum_bytes), ("cum_rbs", cum_rbs)):
            if val is not None:
                getattr(self, name)[...] = np.asarray(val).reshape(getattr(self, name).shape)

    def get_state(self):
        return {k: getattr(self, k).copy() for k in
                ("avg_rate", "tx_bytes", "slice_offset", "nvs_ewma", "cum_bytes", "cum_rbs")}

    def step(self, cqi, rand2=None, dt=0.001, active=None, want_aux=False, queue=None, hol=None):
        """One TTI.  cqi: uint8 [B][U][G] (or [B][U][R]); rand2: int32 [B][2]."""
        B, U, S, G = self.B, self.U, self.S, self.G
        cqi = np.ascontiguousarray(cqi, dtype=np.uint8)
        assert cqi.size == B * U * (self.R if self.cqi_per_rb else G), cqi.shape
        if rand2 is None:
            rand2 = np.zeros((B, 2), dtype=np.int32)
        rand2 = np.ascontiguousarray(rand2, dtype=np.int32).reshape(B, -1)   # [B][2]; id 11: [B][300 * users]
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8).reshape(B, U)
        per = (B, U) if self.nb == 1 else (B, U, 2)
        q = None if queue is None else np.ascontiguousarray(queue, dtype=np.int32).reshape(per)
        h = None if hol is None else np.ascontiguousarray(hol, dtype=np.float64).reshape(per)
        out = {
            "rbg_to_ue": np.empty((B, G), dtype=np.int16),
            "tbs_bits": np.empty((B, U), dtype=np.int32),
            "mcs": np.empty((B, U), dtype=np.uint8),
        }
        aux = {}
        if want_aux:
            aux = {
                "final_cqi": np.empty((B, U), dtype=np.uint8),
                "slice_target": np.empty((B, S), dtype=np.int32),
                "slice_quota": np.empty((B, S), dtype=np.int32),
                "nvs_slice": np.empty((B,), dtype=np.int32),
            }
            if self.algo == 10:
                L = self.grant_list_len
                aux.update({"alloc_n": np.empty((B,), dtype=np.int32), "alloc_ue": np.empty((B, L), dtype=np.int16),
                            "alloc_rbg": np.empty((B, L), dtype=np.int16)})
        io = _Io(_ptr(self.avg_rate), _ptr(self.tx_bytes), _ptr(self.cum_bytes), _ptr(self.cum_rbs),
                 _ptr(self.slice_offset), _ptr(self.nvs_ewma),
                 _ptr(cqi), _ptr(act), _ptr(rand2), float(dt),
                 _ptr(out["rbg_to_ue"]), _ptr(out["tbs_bits"]), _ptr(out["mcs"]), _ptr(aux.get("final_cqi")),
                 _ptr(aux.get("slice_target")), _ptr(aux.get("slice_quota")), _ptr(aux.get("nvs_slice")),
                 _ptr(aux.get("alloc_n")), _ptr(aux.get("alloc_ue")), _ptr(aux.get("alloc_rbg")),
                 int(rand2.shape[1]), _ptr(q), _ptr(h), self.grant_list_len)
        rc = lib().rso_step(C.byref(self._cfg), B, C.byref(io), self.n_threads)
        if rc != 0:
            raise RuntimeError(f"rso_step failed: {rc}")
        out.update(aux)
        return out


def std_sort_desc(keys) -> np.ndarray:
    keys = np.ascontiguousarray(keys, dtype=np.float64)
    perm = np.empty(keys.shape[0], dtype=np.int32)
    lib().rso_std_sort_desc(_ptr(keys), keys.shape[0], _ptr(perm))
    return perm


def introsort_emul_desc(keys, depth_limit=-1) -> np.ndarray:
    keys = np.ascontiguousarray(keys, dtype=np.float64)
    perm = np.empty(keys.shape[0], dtype=np.int32)
    lib().rso_introsort_emul_desc(_ptr(keys), keys.shape[0], int(depth_limit), _ptr(perm))
    return perm

"""CPU: the NCCL companion library exports the entry point include/rs_sched_nccl_buffers.h declares (loads without a
GPU; no calls made), and that header adds to rs_sched_nccl.h without redeclaring any of its entry points."""
import ctypes
import os
import re

from tests.helpers import ROOT


def _declared(name):
    src = open(os.path.join(ROOT, "include", name)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", src)))


def test_nccl_buffers_header_symbols_are_exported():
    import torch  # noqa: F401  -- before the library: a process that loads the system libnccl first cannot import torch later
    names = _declared("rs_sched_nccl_buffers.h")
    assert names == ["rs_reduce_buffer_stats"]
    assert not set(names) & set(_declared("rs_sched_nccl.h"))
    path = os.path.join(ROOT, "radiosaber_b200", "librs_nccl.so")
    assert os.path.exists(path), "build with make -C radiosaber_b200/csrc"
    L = ctypes.CDLL(path)
    for name in names:
        assert hasattr(L, name), name

"""Test harness: memory spaces + loaders for the three implementations of the C ABI.

TEST INFRASTRUCTURE ONLY.  Nothing under aresdb_b200/ imports this module or anything
under oracle/.
"""
from __future__ import annotations

import ctypes as C
import functools
from pathlib import Path

import numpy as np
import pytest

from aresdb_b200 import cabi

ROOT = Path(__file__).resolve().parent.parent
REF_DIR = ROOT / "oracle" / "_ref"
ORACLE_LIB = ROOT / "oracle" / "build" / "liboracle.so"


from aresdb_b200.memory import Buf, CudaSpace, HostSpace  # noqa: E402,F401


class Backend:
    def __init__(self, name: str, lib: cabi.Library, space):
        self.name, self.lib, self.space = name, lib, space
        self.is_gpu = isinstance(space, CudaSpace)

    # convenience
    @property
    def device(self):
        return self.space.device

    def put(self, data) -> Buf:
        return self.space.put(data)

    def zeros(self, nbytes) -> Buf:
        return self.space.zeros(nbytes)


@functools.lru_cache(maxsize=None)
def get_backend(name: str) -> Backend:
    if name == "ref":
        alg, mem = REF_DIR / "libalgorithm.so", REF_DIR / "libmem_ref.so"
        if not alg.exists():
            pytest.skip("oracle/_ref not built (ARESDB_REFERENCE=<reference tree> bash oracle/build_ref.sh)")
        return Backend("ref", cabi.Library(alg, mem, has_plan_api=False, name="ref"), HostSpace())
    if name == "oracle":
        if not ORACLE_LIB.exists():
            import subprocess, sys
            subprocess.run([sys.executable, str(ROOT / "oracle" / "build_oracle.py")], check=True)
        return Backend("oracle", cabi.Library(ORACLE_LIB, None, has_plan_api=False, name="oracle"), HostSpace())
    if name == "b200":
        import torch
        if not torch.cuda.is_available():
            pytest.skip("no CUDA device")
        lib = cabi.load_engine()
        torch.zeros(1, device="cuda:0")  # create the context before the first C-ABI call
        return Backend("b200", lib, CudaSpace(0))
    raise KeyError(name)


# ---- column / vector builders shared by the tests ---------------------------------------------
from aresdb_b200.columns import NP_OF as _NP_OF, pack_bits  # noqa: E402,F401
from aresdb_b200 import columns as _columns  # noqa: E402


def align(n: int, a: int = 8) -> int:
    return (n + a - 1) // a * a


def make_column(be, data_type, values, valid=None, counts=None, start_bit=0, default=None, value_align=64):
    return _columns.make_column(be.space, data_type, values, valid, counts, start_bit, default, value_align)


def make_scratch(be: Backend, data_type: int, values, valid):
    """Scratch-space vector: values (4 B each) followed, 8-byte aligned, by bool bytes."""
    vb = np.ascontiguousarray(values, dtype=_NP_OF[data_type]).view(np.uint8).reshape(-1)
    nulls_off = align(vb.size, 8)
    raw = np.zeros(nulls_off + len(valid), np.uint8)
    raw[:vb.size] = vb
    raw[nulls_off:] = np.asarray(valid, dtype=np.uint8)
    buf = be.put(raw)
    return buf, nulls_off


def dim_layout(num_dims_per_width, capacity: int):
    """(value offsets, null offsets, total bytes) of a DimensionVector block
    (reference query/common/dimval.go:122-145)."""
    offs, pos = [], 0
    widths = []
    for w, cnt in zip(cabi.DIM_WIDTHS, num_dims_per_width):
        for _ in range(cnt):
            offs.append(pos)
            widths.append(w)
            pos += w * capacity
    nulls = []
    for _ in widths:
        nulls.append(pos)
        pos += capacity
    return offs, nulls, widths, pos

"""ctypes binding of oracle/c/b9_oracle.c (TEST INFRASTRUCTURE; see that file's header)."""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import List, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "build", "libb9oracle.so")

COMPLETE, ERROR, REJECTED, UNSUPPORTED = 0, 1, 3, 4
HANDLER_IDS = {"identity": 0, "echo": 0, "crc32": 1, "vadd_f32": 2, "json_sum": 3}
STATUS_NAMES = {0: "COMPLETE", 1: "ERROR", 3: "REJECTED", 4: "UNSUPPORTED"}

DEFAULT_NOW_NS = 1_789_970_992_573_161_412
DEFAULT_WS = "ws-b200"
DEFAULT_STUB = "7f1c2d3e-4a5b-4c6d-8e9f-0a1b2c3d4e5f"


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "c", "b9_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", os.path.join(_HERE, "c"), "-s"])
    return _SO


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
        _lib.b9o_run_batch.restype = ctypes.c_int64
        _lib.b9o_run_batch.argtypes = [
            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int,
            ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int32, ctypes.c_uint32, ctypes.c_int64,
            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int]
        _lib.b9o_task_queue_scale.restype = ctypes.c_int
        _lib.b9o_task_queue_scale.argtypes = [ctypes.c_int64] * 4 + [ctypes.POINTER(ctypes.c_int)]
    return _lib


class OracleResult:
    def __init__(self, status, has, offsets, payload, wire_offsets=None, wire=None, handler=None):
        self.handler = handler        # the handler name the batch ran
        self.status = status          # uint8 [n]
        self.has = has                # uint8 [n]
        self.offsets = offsets        # uint64 [n+1]
        self.payload = payload        # uint8 [total]
        self.wire_offsets = wire_offsets
        self.wire = wire

    def result(self, i: int) -> Optional[bytes]:
        if not self.has[i]:
            return None
        return self.payload[int(self.offsets[i]):int(self.offsets[i + 1])].tobytes()

    def wire_msg(self, i: int) -> bytes:
        return self.wire[int(self.wire_offsets[i]):int(self.wire_offsets[i + 1])].tobytes()


def run_batch(task_ids: np.ndarray, payload: np.ndarray, offsets: np.ndarray, handler: str,
              nthreads: int = 1, keep_wire: bool = False, out_cap: Optional[int] = None,
              now_ns: int = DEFAULT_NOW_NS, workspace: str = DEFAULT_WS, stub: str = DEFAULT_STUB,
              max_retries: int = 3, timeout: int = 3600, ttl: int = 7200) -> OracleResult:
    n = int(offsets.shape[0] - 1)
    ids = np.ascontiguousarray(task_ids, dtype=np.uint8)
    pl = np.ascontiguousarray(payload, dtype=np.uint8)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    if out_cap is None:
        out_cap = int(pl.size) * 6 + 64 * n + 64
    status = np.zeros(n, np.uint8)
    has = np.zeros(n, np.uint8)
    out_off = np.zeros(n + 1, np.uint64)
    out = np.empty(out_cap, np.uint8)
    w_off = w = None
    w_cap = 0
    if keep_wire:
        w_cap = int(pl.size) * 6 + 512 * n + 64
        w_off = np.zeros(n + 1, np.uint64)
        w = np.empty(w_cap, np.uint8)
    total = lib().b9o_run_batch(
        ids.ctypes.data, pl.ctypes.data, off.ctypes.data, n, HANDLER_IDS[handler],
        workspace.encode(), stub.encode(), max_retries, timeout, ttl, now_ns,
        status.ctypes.data, has.ctypes.data, out_off.ctypes.data, out.ctypes.data, out_cap,
        w_off.ctypes.data if keep_wire else None, w.ctypes.data if keep_wire else None, w_cap, nthreads)
    if total < 0:
        raise MemoryError("oracle output capacity too small")
    if keep_wire:
        w = w[:int(w_off[-1])]
    return OracleResult(status, has, out_off, out[:total], w_off, w, handler)


def task_queue_scale(q: int, tpc: int, max_containers: int, max_replicas: int) -> Tuple[int, bool]:
    v = ctypes.c_int(0)
    d = lib().b9o_task_queue_scale(q, tpc, max_containers, max_replicas, ctypes.byref(v))
    return d, bool(v.value)

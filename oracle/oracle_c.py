"""ctypes binding of the C oracle (oracle/egs_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Builds oracle/_build/libegs_oracle.so with gcc on first use when it is missing.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libegs_oracle.so")


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "egs_oracle.c")
    hdr = os.path.join(_HERE, "egs_oracle.h")
    stale = (not os.path.exists(_SO)) or any(
        os.path.getmtime(p) > os.path.getmtime(_SO) for p in (src, hdr))
    if force or stale:
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-g", "-std=c11", "-fPIC", "-pthread", "-shared",
                               "-o", _SO, src])
    return _SO


class Unit(C.Structure):
    _fields_ = [("core", C.c_int64), ("mem", C.c_int64), ("count", C.c_int64)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        L = _lib
        L.egso_create.restype = C.c_void_p
        L.egso_create.argtypes = [C.c_int, C.c_int]
        L.egso_destroy.argtypes = [C.c_void_p]
        L.egso_add_node.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
        L.egso_num_nodes.argtypes = [C.c_void_p]
        L.egso_gpu_count.argtypes = [C.c_void_p, C.c_int]
        L.egso_set_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.egso_get_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.egso_request_hash.argtypes = [C.c_int, C.c_void_p, C.c_char_p]
        L.egso_unit_from_requests.argtypes = [C.c_int64, C.c_int64, C.c_void_p]
        L.egso_trade.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.egso_filter.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.egso_score.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.egso_bind.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.egso_peek.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.egso_add_pod.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.egso_forget_pod.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.egso_cache_load.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.egso_cache_dump.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.egso_known_pod.argtypes = [C.c_void_p, C.c_uint64]
        L.egso_released_pod.argtypes = [C.c_void_p, C.c_uint64]
        L.egso_schedule_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int] + \
            [C.c_void_p] * 6 + [C.c_int, C.c_void_p, C.c_void_p]
        L.egso_mix64.restype = C.c_uint64
        L.egso_mix64.argtypes = [C.c_uint64]
        L.egso_sha256.argtypes = [C.c_char_p, C.c_uint64, C.c_void_p]
    return _lib


def _units(req: Sequence[Tuple[int, int, int]]):
    arr = (Unit * max(1, len(req)))()
    for i, (c, m, k) in enumerate(req):
        arr[i].core, arr[i].mem, arr[i].count = c, m, k
    return arr


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _alloc_arrays(alloc):
    off = [0]
    idx: List[int] = []
    for a in alloc:
        a = a or []
        idx.extend(a)
        off.append(len(idx))
    return np.array(off, dtype=np.int32), np.array(idx + [0], dtype=np.int32)


def _alloc_lists(off, idx, Cn):
    return [[int(idx[k]) for k in range(off[c], off[c + 1])] for c in range(Cn)]


class OracleC:
    """Thin object wrapper; method names follow oracle/egs_oracle.py's Scheduler."""

    def __init__(self, policy: int, faithful: bool = False):
        self.L = lib()
        self.h = self.L.egso_create(policy, 1 if faithful else 0)

    def __del__(self):
        try:
            self.L.egso_destroy(self.h)
        except Exception:
            pass

    def add_node(self, core_alloc: int, mem_alloc: int) -> int:
        return self.L.egso_add_node(self.h, core_alloc, mem_alloc)

    @property
    def n_nodes(self) -> int:
        return self.L.egso_num_nodes(self.h)

    def gpu_count(self, node: int) -> int:
        return self.L.egso_gpu_count(self.h, node)

    def set_rows(self, node: int, core, mem) -> None:
        c = np.ascontiguousarray(core, dtype=np.int64)
        m = np.ascontiguousarray(mem, dtype=np.int64)
        self.L.egso_set_rows(self.h, node, _ptr(c), _ptr(m))

    def rows(self, node: int):
        g = self.gpu_count(node)
        c = np.zeros(max(g, 1), dtype=np.int64)
        m = np.zeros(max(g, 1), dtype=np.int64)
        self.L.egso_get_rows(self.h, node, _ptr(c), _ptr(m))
        return [(int(c[i]), int(m[i])) for i in range(g)]

    def trade(self, node: int, req):
        off = np.zeros(len(req) + 1, dtype=np.int32)
        idx = np.zeros(len(req) * 16 + 1, dtype=np.int32)
        sc = C.c_int64(0)
        st = self.L.egso_trade(self.h, node, len(req), _units(req), _ptr(off), _ptr(idx), C.byref(sc))
        if st != 0:
            return None
        return _alloc_lists(off, idx, len(req)), sc.value

    def filter(self, node_ids, req, threads: int = 1) -> np.ndarray:
        ids = None if node_ids is None else np.ascontiguousarray(node_ids, dtype=np.int32)
        n = self.n_nodes if ids is None else len(ids)
        out = np.zeros(max(n, 1), dtype=np.uint8)
        self.L.egso_filter(self.h, n, _ptr(ids), len(req), _units(req), threads, _ptr(out))
        return out[:n]

    def score(self, node_ids, req):
        ids = None if node_ids is None else np.ascontiguousarray(node_ids, dtype=np.int32)
        n = self.n_nodes if ids is None else len(ids)
        out = np.zeros(max(n, 1), dtype=np.int64)
        st = self.L.egso_score(self.h, n, _ptr(ids), len(req), _units(req), _ptr(out))
        return st, out[:n]

    def bind(self, node: int, req, uid: int):
        off = np.zeros(len(req) + 1, dtype=np.int32)
        idx = np.zeros(len(req) * 16 + 1, dtype=np.int32)
        st = self.L.egso_bind(self.h, node, len(req), _units(req), uid, _ptr(off), _ptr(idx))
        return st, (_alloc_lists(off, idx, len(req)) if st == 0 else None)

    def peek(self, node: int, req):
        off = np.zeros(len(req) + 1, dtype=np.int32)
        idx = np.zeros(len(req) * 16 + 1, dtype=np.int32)
        sc = C.c_int64(0)
        ok = self.L.egso_peek(self.h, node, len(req), _units(req), C.byref(sc), _ptr(off), _ptr(idx))
        if not ok:
            return None
        return _alloc_lists(off, idx, len(req)), sc.value

    def add_pod(self, node: int, req, alloc, uid: int) -> int:
        off, idx = _alloc_arrays(alloc)
        return self.L.egso_add_pod(self.h, node, len(req), _units(req), _ptr(off), _ptr(idx), uid)

    def forget_pod(self, node: int, req, alloc, uid: int) -> int:
        off, idx = _alloc_arrays(alloc)
        return self.L.egso_forget_pod(self.h, node, len(req), _units(req), _ptr(off), _ptr(idx), uid)

    def cache_load(self, req, valid, score, alloc_mask) -> int:
        """Install cached options of shape `req` on nodes 0..n-1 (state of a scheduler that already ran)."""
        v = np.ascontiguousarray(valid, dtype=np.uint8)
        sc = np.ascontiguousarray(score, dtype=np.int64)
        am = np.ascontiguousarray(alloc_mask, dtype=np.uint8)
        return self.L.egso_cache_load(self.h, len(req), _units(req), len(v), None, _ptr(v), _ptr(sc), _ptr(am))

    def cache_dump(self, req, n: Optional[int] = None):
        """Option cache of request `req` on nodes [0, n): (valid u8[n], score i64[n], alloc_mask u8[n, 4]) --
        egso_peek of every node in one call, laid out like egso_cache_load's input."""
        n = self.n_nodes if n is None else n
        v = np.zeros(max(n, 1), np.uint8); sc = np.zeros(max(n, 1), np.int64); am = np.zeros((max(n, 1), 4), np.uint8)
        st = self.L.egso_cache_dump(self.h, len(req), _units(req), n, _ptr(v), _ptr(sc), _ptr(am))
        if st != 0:
            raise ValueError(f"egso_cache_dump: status {st}")
        return v[:n], sc[:n], am[:n]

    def known_pod(self, uid: int) -> bool:
        return bool(self.L.egso_known_pod(self.h, uid))

    def released_pod(self, uid: int) -> bool:
        return bool(self.L.egso_released_pod(self.h, uid))

    def schedule_batch(self, c_off: np.ndarray, units: np.ndarray, uids: Optional[np.ndarray] = None,
                       threads: int = 1, vec_pods: int = 0):
        """units: int64 [sum C][3]; returns dict of numpy arrays."""
        P = len(c_off) - 1
        N = self.n_nodes
        c_off = np.ascontiguousarray(c_off, dtype=np.int32)
        units = np.ascontiguousarray(units, dtype=np.int64)
        out = dict(node=np.zeros(P, np.int32), status=np.zeros(P, np.int32),
                   alloc_mask=np.zeros((P, 4), np.uint8), fit_count=np.zeros(P, np.int32),
                   fit_digest=np.zeros(P, np.uint64), score_digest=np.zeros(P, np.uint64))
        vf = np.zeros((vec_pods, N), np.uint8) if vec_pods else None
        vs = np.zeros((vec_pods, N), np.int32) if vec_pods else None
        u = None if uids is None else np.ascontiguousarray(uids, dtype=np.uint64)
        self.L.egso_schedule_batch(self.h, P, _ptr(c_off), _ptr(units), _ptr(u), threads,
                                   _ptr(out["node"]), _ptr(out["status"]), _ptr(out["alloc_mask"]),
                                   _ptr(out["fit_count"]), _ptr(out["fit_digest"]), _ptr(out["score_digest"]),
                                   vec_pods, _ptr(vf), _ptr(vs))
        if vec_pods:
            out["vec_fit"], out["vec_score"] = vf, vs
        return out


def request_hash(req) -> str:
    buf = C.create_string_buffer(9)
    lib().egso_request_hash(len(req), _units(req), buf)
    return buf.value.decode()


def sha256(msg: bytes) -> bytes:
    out = (C.c_uint8 * 32)()
    lib().egso_sha256(msg, len(msg), out)
    return bytes(out)


def unit_from_requests(core: int, mem: int):
    u = Unit()
    lib().egso_unit_from_requests(core, mem, C.byref(u))
    return (u.core, u.mem, u.count)

"""ctypes loader for the CPU oracle (oracle/gcra_oracle.cpp).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package
(throttlecrab_b200/) must never import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgcra_oracle.so")

REQ_DTYPE = np.dtype([("key", "<u8"), ("max_burst", "<i8"), ("count_per_period", "<i8"),
                      ("period", "<i8"), ("quantity", "<i8"), ("now_ns", "<i8")])
RES_DTYPE = np.dtype([("remaining", "<i8"), ("reset_after_ns", "<i8"), ("retry_after_ns", "<i8"),
                      ("status", "<i4"), ("allowed", "u1"), ("pad", "u1", (3,))])
assert REQ_DTYPE.itemsize == 48 and RES_DTYPE.itemsize == 32

PERIODIC, PROBABILISTIC, ADAPTIVE = 0, 1, 2


def build(force=False):
    src = [os.path.join(_HERE, f) for f in ("gcra_oracle.cpp", "gcra_oracle.h")]
    if force or not os.path.exists(_SO) or any(
            os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_SO) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libgcra_oracle.so"],
                              stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):      # loading never recompiles a built library: the tree may be read-only
            build()
        L = C.CDLL(_SO)
        vp, u64, i64, cp = C.c_void_p, C.c_uint64, C.c_int64, C.c_char_p
        L.ora_create.restype = vp
        L.ora_create.argtypes = [C.c_int, u64, i64, u64, u64, u64]
        L.ora_destroy.argtypes = [vp]
        L.ora_get.argtypes = [vp, cp, u64, i64, C.POINTER(i64)]
        L.ora_cas.argtypes = [vp, cp, u64, i64, i64, u64, i64]
        L.ora_set_nx.argtypes = [vp, cp, u64, i64, u64, i64]
        L.ora_derive.argtypes = [i64, i64, i64, C.POINTER(i64), C.POINTER(i64)]
        L.ora_rate_limit.argtypes = [vp, cp, u64, i64, i64, i64, i64, i64, vp]
        L.ora_replay.argtypes = [vp, u64, vp, vp]
        L.ora_replay_sharded.restype = C.c_double
        L.ora_replay_sharded.argtypes = [vp, C.c_int, u64, vp, vp]
        for f in ("ora_len", "ora_expired_count", "ora_sweeps"):
            getattr(L, f).restype = u64
            getattr(L, f).argtypes = [vp]
        L.ora_entry.argtypes = [vp, cp, u64, C.POINTER(i64), C.POINTER(i64)]
        L.ora_force_sweep.restype = u64
        L.ora_force_sweep.argtypes = [vp, i64]
        _lib = L
    return _lib


def _kb(key):
    return key.encode("utf-8") if isinstance(key, str) else bytes(key)


def derive(max_burst, count, period):
    ei, dvt = C.c_int64(), C.c_int64()
    st = lib().ora_derive(max_burst, count, period, C.byref(ei), C.byref(dvt))
    return st, ei.value, dvt.value


class OracleStore:
    """One reference store (Periodic / Probabilistic / Adaptive) + the RateLimiter over it."""

    def __init__(self, kind=ADAPTIVE, capacity=1000, created_ns=0, p0=0, p1=0, p2=0):
        self._h = lib().ora_create(kind, capacity, created_ns, p0, p1, p2)
        self.kind = kind

    def close(self):
        if self._h:
            lib().ora_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # Store trait
    def get(self, key, now_ns):
        k = _kb(key)
        v = C.c_int64()
        return v.value if lib().ora_get(self._h, k, len(k), now_ns, C.byref(v)) else None

    def compare_and_swap_with_ttl(self, key, old, new, ttl_ns, now_ns):
        k = _kb(key)
        return bool(lib().ora_cas(self._h, k, len(k), old, new, ttl_ns, now_ns))

    def set_if_not_exists_with_ttl(self, key, value, ttl_ns, now_ns):
        k = _kb(key)
        return bool(lib().ora_set_nx(self._h, k, len(k), value, ttl_ns, now_ns))

    # RateLimiter::rate_limit -> (status, allowed, remaining, reset_after_ns, retry_after_ns)
    def rate_limit(self, key, max_burst, count, period, quantity, now_ns):
        k = _kb(key)
        out = np.zeros(1, RES_DTYPE)
        lib().ora_rate_limit(self._h, k, len(k), max_burst, count, period, quantity, now_ns,
                             out.ctypes.data)
        r = out[0]
        return (int(r["status"]), bool(r["allowed"]), int(r["remaining"]),
                int(r["reset_after_ns"]), int(r["retry_after_ns"]))

    def replay(self, req):
        """req: REQ_DTYPE array whose `key` column holds key ids (key string "k:<id>")."""
        req = np.ascontiguousarray(req, REQ_DTYPE)
        out = np.zeros(len(req), RES_DTYPE)
        lib().ora_replay(self._h, len(req), req.ctypes.data, out.ctypes.data)
        return out

    def len(self):
        return int(lib().ora_len(self._h))

    def expired_count(self):
        return int(lib().ora_expired_count(self._h))

    def sweeps(self):
        return int(lib().ora_sweeps(self._h))

    def entry(self, key):
        k = _kb(key)
        t, e = C.c_int64(), C.c_int64()
        if lib().ora_entry(self._h, k, len(k), C.byref(t), C.byref(e)):
            return t.value, e.value
        return None

    def force_sweep(self, now_ns):
        return int(lib().ora_force_sweep(self._h, now_ns))


def replay_sharded(stores, req):
    """Time the decision loops of `len(stores)` hash-sharded stores (threads). Returns (out, seconds)."""
    req = np.ascontiguousarray(req, REQ_DTYPE)
    out = np.zeros(len(req), RES_DTYPE)
    arr = (C.c_void_p * len(stores))(*[s._h for s in stores])
    sec = lib().ora_replay_sharded(arr, len(stores), len(req), req.ctypes.data, out.ctypes.data)
    return out, sec

"""The oracle's entry points for a float signal (test infrastructure only): getevents(n, pa, rna) as orc_getevents
restates it, and create_events from given prefix sums (orc_events). Used by the tests of the pA-input path."""
from __future__ import annotations

import ctypes as C

import numpy as np

_u64p = C.POINTER(C.c_uint64)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)


def _p(a, t):
    return a.ctypes.data_as(t)


def _bind(orc):
    L = orc.lib
    L.orc_getevents.restype = C.c_int64
    L.orc_getevents.argtypes = [C.c_uint64, _f32p, C.c_int, C.c_uint64, _u64p, _f32p, _f32p, _f32p]
    L.orc_events.restype = C.c_uint64
    L.orc_events.argtypes = [_u64p, C.c_uint64, _f64p, _f64p, C.c_uint64, _u64p, _f32p, _f32p, _f32p]
    return L


def getevents_pa(orc, pa, rna=0):
    """getevents(n, pa, rna) (events.c:553-573) on a float array -> (start u64, length f32, mean f32, stdv f32)"""
    L = _bind(orc)
    pa = np.ascontiguousarray(pa, dtype=np.float32)
    n = pa.shape[0]
    cap = n // 2 + 4
    st = np.empty(cap, dtype=np.uint64)
    ln, mn, sd = (np.empty(cap, dtype=np.float32) for _ in range(3))
    ne = L.orc_getevents(n, _p(pa, _f32p), int(rna), cap, _p(st, _u64p), _p(ln, _f32p), _p(mn, _f32p), _p(sd, _f32p))
    assert ne >= 0, ne
    return st[:ne].copy(), ln[:ne].copy(), mn[:ne].copy(), sd[:ne].copy()


def events_from_prefix(orc, peaks, S, Q):
    """create_events (events.c:457-504) from peak positions and the prefix sums S, Q (n+1 entries each)"""
    L = _bind(orc)
    peaks = np.ascontiguousarray(peaks, dtype=np.uint64)
    S = np.ascontiguousarray(S, dtype=np.float64)
    Q = np.ascontiguousarray(Q, dtype=np.float64)
    n = S.shape[0] - 1
    cap = n // 2 + 4
    st = np.empty(cap, np.uint64)
    ln, mn, sd = (np.empty(cap, np.float32) for _ in range(3))
    ne = L.orc_events(_p(peaks, _u64p), peaks.shape[0], _p(S, _f64p), _p(Q, _f64p), n, _p(st, _u64p), _p(ln, _f32p),
                      _p(mn, _f32p), _p(sd, _f32p))
    return st[:ne].copy(), ln[:ne].copy(), mn[:ne].copy(), sd[:ne].copy()

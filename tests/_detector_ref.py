"""The streaming reference of live event detection for any detector set (sgpu_set_detector), built from the oracle's
stage-level entry points (test infrastructure only).

It is _live_ref.stream_reference with two generalisations: the detector_param may be given (params), and after chunk
k of a read (n_k samples so far) the detector is stepped over the positions [stepped, n_k - max(w_short, w_long) + 1),
the positions whose t-statistics the later samples cannot change for either window. For the reference's sets
(w_long > w_short) that is _live_ref's rule, n_k - w_long + 1. END steps the rest. Every peak emitted during those
steps closes one event, and the chunk reports those events; END also reports the last one."""
from __future__ import annotations

import ctypes as C

import numpy as np

from _oracle_pa import events_from_prefix

_f32p = C.POINTER(C.c_float)
_u64p = C.POINTER(C.c_uint64)


def stream_reference(orc, pa, rna, chunks, thr_long=None, params=None):
    """-> (the events each chunk reports as (start u64, length f32, mean f32, stdv f32), the emitted peaks as
    (position, chunk) pairs); the last chunk ends the read. params: a detector_param (w_short, w_long, thr_short,
    thr_long, peak_height) used instead of the reference's set for rna"""
    pa = np.ascontiguousarray(pa, dtype=np.float32)
    n = pa.shape[0]
    assert sum(chunks) == n
    S, Q = orc.prefix(pa)
    p = orc.params(rna) if params is None else orc.Params(*params)
    if thr_long is not None:
        p.thr_long = float(thr_long)
    t1 = np.ascontiguousarray(orc.tstat(S, Q, p.w_short), dtype=np.float32)
    t2 = np.ascontiguousarray(orc.tstat(S, Q, p.w_long), dtype=np.float32)
    if n == 0:
        t1 = t2 = np.zeros(1, np.float32)
    s, l = orc.Det(), orc.Det()
    orc.lib.orc_det_init(C.byref(s), C.byref(l))
    buf = np.empty(max(n, 1) * 2 + 4, np.uint64)
    w = max(p.w_short, p.w_long)
    peaks, closed = [], []  # every valid peak with its chunk; number of events closed after each chunk
    stepped, have = 0, 0
    for k, m in enumerate(chunks):
        have += m
        to = have if k == len(chunks) - 1 else max(stepped, have - w + 1)
        if to > stepped:
            np_ = orc.lib.orc_detect(t1.ctypes.data_as(_f32p), t2.ctypes.data_as(_f32p), stepped, to, C.byref(p),
                                     C.byref(s), C.byref(l), buf.ctypes.data_as(_u64p), buf.shape[0])
            peaks += [(int(q), k) for q in buf[:np_] if 0 < int(q) < n]  # events.c:481-485
            stepped = to
        closed.append(len(peaks))
    if n == 0:
        e = np.empty(0, np.float32)
        return [(np.empty(0, np.uint64), e, e, e) for _ in chunks], peaks
    ev = events_from_prefix(orc, np.array([q for q, _ in peaks], np.uint64), S, Q)
    out, a = [], 0
    for k in range(len(chunks)):
        b = closed[k] + (1 if k == len(chunks) - 1 else 0)
        out.append(tuple(x[a:b] for x in ev))
        a = b
    return out, peaks


def whole_read(orc, pa, rna, thr_long=None, params=None):
    """getevents on the whole read with the given long threshold or detector_param (a read of 0 samples: no event)"""
    return stream_reference(orc, pa, rna, [len(pa)], thr_long, params)[0][0]

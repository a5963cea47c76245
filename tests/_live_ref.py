"""The streaming reference of live event detection (include/sigtk_b200.h, "live event detection"), built from the
oracle's stage-level entry points (test infrastructure only).

After chunk k of a read (n_k samples so far) the detector is stepped, with states carried from chunk to chunk, over
the positions [stepped, n_k - w2 + 1); END steps the rest. Every peak emitted during those steps closes one event, and
the chunk reports those events; END also reports the last one. The t-statistics are those of the whole read: the
positions stepped after chunk k are exactly those whose t-statistics the later samples cannot change."""
from __future__ import annotations

import ctypes as C

import numpy as np

from _oracle_pa import events_from_prefix

_f32p = C.POINTER(C.c_float)
_u64p = C.POINTER(C.c_uint64)


def split_lengths(n, rng, w2=14):
    """a seeded random split of n samples into chunks: 1-sample chunks, chunks shorter than w2, long ones; sometimes
    an empty chunk at the end (END in an entry of its own)"""
    out, left = [], n
    while left > 0:
        u = rng.random()
        k = 1 if u < 0.15 else int(rng.integers(2, w2)) if u < 0.45 else int(rng.integers(w2, 3000))
        k = min(k, left)
        out.append(k)
        left -= k
    if not out or rng.random() < 0.3:
        out.append(0)
    return out


def stream_reference(orc, pa, rna, chunks, thr_long=None):
    """-> (the events each chunk reports as (start u64, length f32, mean f32, stdv f32), the emitted peaks as
    (position, chunk) pairs); the last chunk ends the read"""
    pa = np.ascontiguousarray(pa, dtype=np.float32)
    n = pa.shape[0]
    assert sum(chunks) == n
    S, Q = orc.prefix(pa)
    p = orc.params(rna)
    if thr_long is not None:
        p.thr_long = float(thr_long)
    t1 = np.ascontiguousarray(orc.tstat(S, Q, p.w_short), dtype=np.float32)
    t2 = np.ascontiguousarray(orc.tstat(S, Q, p.w_long), dtype=np.float32)
    if n == 0:
        t1 = t2 = np.zeros(1, np.float32)
    s, l = orc.Det(), orc.Det()
    orc.lib.orc_det_init(C.byref(s), C.byref(l))
    buf = np.empty(max(n, 1) * 2 + 4, np.uint64)
    peaks, closed = [], []  # every valid peak with its chunk; number of events closed after each chunk
    stepped, have = 0, 0
    for k, m in enumerate(chunks):
        have += m
        to = have if k == len(chunks) - 1 else max(stepped, have - p.w_long + 1)
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


def whole_read(orc, pa, rna, thr_long=None):
    """getevents on the whole read with the given long threshold (a read of 0 samples: no event)"""
    return stream_reference(orc, pa, rna, [len(pa)], thr_long)[0][0]


def concat(tables):
    return tuple(np.concatenate([t[j] for t in tables]) for j in range(4))


def same_events(a, b):
    """two (start, length, mean, stdv) tuples, every float by its bits"""
    return (np.array_equal(np.asarray(a[0], np.uint64), np.asarray(b[0], np.uint64)) and
            all(np.array_equal(np.asarray(a[j], np.float32).view(np.uint32), np.asarray(b[j], np.float32).view(np.uint32))
                for j in (1, 2, 3)))

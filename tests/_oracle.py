"""ctypes loaders for the two CHECKERS (test infrastructure only):

  oracle/liboracle.so          our CPU restatement (oracle/sigtk_oracle.c)
  oracle/_ref/libsigtk_ref.so  the unmodified reference functions (oracle/ref_shim.c + /root/reference sources)

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libsigtk_ref.so")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "sigtk")

_u64p = C.POINTER(C.c_uint64)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_i16p = C.POINTER(C.c_int16)


def _p(a, t):
    return a.ctypes.data_as(t)


def build_oracle():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
            os.path.join(ORACLE_DIR, "sigtk_oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "liboracle.so"], stdout=subprocess.DEVNULL)


class _EventLib:
    """Common surface of both checkers: pa / event_read / stat / time_events."""

    def __init__(self, path: str, prefix: str):
        self.lib = C.CDLL(path)
        self._sym_prefix = prefix
        g = lambda n: getattr(self.lib, prefix + n)
        self._pa = g("pa")
        self._pa.argtypes = [_i16p, C.c_uint64, C.c_double, C.c_double, C.c_double, _f32p]
        self._ev = g("event_read")
        self._ev.restype = C.c_int64
        self._ev.argtypes = [_i16p, C.c_uint64, C.c_double, C.c_double, C.c_double, C.c_int, C.c_uint64, _u64p, _f32p,
                             _f32p, _f32p]
        self._stat = g("stat")
        self._stat.argtypes = [_i16p, C.c_uint64, C.c_double, C.c_double, C.c_double, _f32p]
        self._time = g("time_events")
        self._time.restype = C.c_double
        self._time.argtypes = [_i16p, _u64p, C.c_uint64, _f64p, _f64p, _f64p, C.c_int, _u64p]
        self._svb_enc = g("svbzd_encode")
        self._svb_enc.restype = C.c_int64
        self._svb_enc.argtypes = [_i16p, C.c_uint64, C.c_void_p, C.c_uint64]
        self._svb_dec = g("svbzd_decode")
        self._svb_dec.restype = C.c_int64
        self._svb_dec.argtypes = [C.c_void_p, C.c_uint64, _i16p, C.c_uint64]

    def svbzd_encode(self, raw):
        """int16 samples -> the svb-zd stream slow5lib stores in a BLOW5 record (uint8 array)"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        out = np.empty(4 + (raw.shape[0] + 3) // 4 + 4 * raw.shape[0] + 16, dtype=np.uint8)
        n = self._svb_enc(_p(raw, _i16p), raw.shape[0], out.ctypes.data, out.shape[0])
        assert n >= 4, n
        return out[:n].copy()

    def svbzd_decode(self, stream, cap=None):
        """-> int16 samples, or None when the stream is malformed"""
        stream = np.ascontiguousarray(stream, dtype=np.uint8)
        if cap is None:
            cap = int(stream[:4].view(np.uint32)[0]) if stream.shape[0] >= 4 else 0
        out = np.empty(max(cap, 1), dtype=np.int16)
        n = self._svb_dec(stream.ctypes.data, stream.shape[0], _p(out, _i16p), cap)
        return None if n < 0 else out[:n].copy()

    def pa(self, raw, dig, off, rng):
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        out = np.empty(raw.shape[0], dtype=np.float32)
        self._pa(_p(raw, _i16p), raw.shape[0], dig, off, rng, _p(out, _f32p))
        return out

    def events(self, raw, dig, off, rng, rna=0):
        """-> (start u64, length f32, mean f32, stdv f32)"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        n = raw.shape[0]
        cap = n // 2 + 4
        st = np.empty(cap, dtype=np.uint64)
        ln = np.empty(cap, dtype=np.float32)
        mn = np.empty(cap, dtype=np.float32)
        sd = np.empty(cap, dtype=np.float32)
        ne = self._ev(_p(raw, _i16p), n, dig, off, rng, int(rna), cap, _p(st, _u64p), _p(ln, _f32p), _p(mn, _f32p),
                      _p(sd, _f32p))
        assert ne > 0, ne
        return st[:ne].copy(), ln[:ne].copy(), mn[:ne].copy(), sd[:ne].copy()

    def stat(self, raw, dig, off, rng):
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        out = np.empty(6, dtype=np.float32)
        self._stat(_p(raw, _i16p), raw.shape[0], dig, off, rng, _p(out, _f32p))
        return out

    def time_events(self, reads, rna=0):
        """single-thread seconds for pA + event detection over `reads`; -> (seconds, n_samples, n_events)"""
        lens = np.array([r[0].shape[0] for r in reads], dtype=np.uint64)
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        flat = np.concatenate([np.ascontiguousarray(r[0], dtype=np.int16) for r in reads])
        dig = np.array([r[1] for r in reads], dtype=np.float64)
        ofs = np.array([r[2] for r in reads], dtype=np.float64)
        rng = np.array([r[3] for r in reads], dtype=np.float64)
        nev = C.c_uint64(0)
        t = self._time(_p(flat, _i16p), _p(off, _u64p), len(reads), _p(dig, _f64p), _p(ofs, _f64p), _p(rng, _f64p),
                       int(rna), C.byref(nev))
        return float(t), int(off[-1]), int(nev.value)


class Oracle(_EventLib):
    """our CPU restatement, plus its stage-level entry points"""

    def __init__(self):
        build_oracle()
        super().__init__(ORACLE_SO, "orc_")
        L = self.lib

        class Params(C.Structure):
            _fields_ = [("w_short", C.c_uint32), ("w_long", C.c_uint32), ("thr_short", C.c_float),
                        ("thr_long", C.c_float), ("peak_height", C.c_float)]

        class Det(C.Structure):
            _fields_ = [("masked_to", C.c_uint64), ("peak_pos", C.c_int64), ("peak_value", C.c_float),
                        ("valid", C.c_int32)]

        self.Params, self.Det = Params, Det
        L.orc_params.argtypes = [C.c_int, C.POINTER(Params)]
        L.orc_ent.argtypes = [_i16p, C.c_uint64, _f64p]
        L.orc_ent.restype = None
        L.orc_jnn.argtypes = [_i16p, C.c_uint64, C.c_int, C.c_uint64, C.POINTER(C.c_int64)]
        L.orc_jnn.restype = C.c_int64
        L.orc_adaptor_polya_pore.argtypes = [_i16p, C.c_uint64, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                             C.POINTER(C.c_int64), _f32p]
        L.orc_adaptor_polya_pore.restype = None
        L.orc_prefix.argtypes = [_f32p, C.c_uint64, _f64p, _f64p]
        L.orc_tstat.argtypes = [_f64p, _f64p, C.c_uint64, C.c_uint32, _f32p]
        L.orc_det_init.argtypes = [C.POINTER(Det), C.POINTER(Det)]
        L.orc_det_cold.argtypes = [C.POINTER(Det), C.POINTER(Det), C.c_uint64]
        L.orc_detect.restype = C.c_uint64
        L.orc_detect.argtypes = [_f32p, _f32p, C.c_uint64, C.c_uint64, C.POINTER(Params), C.POINTER(Det),
                                 C.POINTER(Det), _u64p, C.c_uint64]

    def ent(self, raw):
        """raw_ent, delta_ent, byte_ent of one record (ent.c:108-151) as float64[3]"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        out = np.zeros(3, dtype=np.float64)
        self.lib.orc_ent(_p(raw, _i16p), raw.shape[0], _p(out, _f64p))
        return out

    def jnn(self, raw, rna=0):
        """segments of `sigtk jnn` for one record (jnn.c:176-282) as int64[k][2]"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        cap = raw.shape[0] // 32 + 2
        xy = np.zeros(2 * cap, dtype=np.int64)
        k = self.lib.orc_jnn(_p(raw, _i16p), raw.shape[0], int(rna), cap, xy.ctypes.data_as(C.POINTER(C.c_int64)))
        assert k >= 0, k
        return xy[:2 * k].reshape(k, 2).copy()

    def adaptor_polya(self, raw, dig, off, rng, rna=0, pore=0):
        """`sigtk prefix` numbers (cfunc.c:169-234) with the adaptor parameters of an R9 pore (pore=0) or of RNA004
        (pore=1, SGPU_PARAM_PORE): -> (pos int64[4], stat float32[6])"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        pos = np.zeros(4, dtype=np.int64)
        st = np.zeros(6, dtype=np.float32)
        self.lib.orc_adaptor_polya_pore(_p(raw, _i16p), raw.shape[0], dig, off, rng, int(rna), int(pore),
                                        pos.ctypes.data_as(C.POINTER(C.c_int64)), _p(st, _f32p))
        return pos, st

    def params(self, rna):
        p = self.Params()
        self.lib.orc_params(int(rna), C.byref(p))
        return p

    def prefix(self, pa):
        pa = np.ascontiguousarray(pa, dtype=np.float32)
        S = np.empty(pa.shape[0] + 1, dtype=np.float64)
        Q = np.empty(pa.shape[0] + 1, dtype=np.float64)
        self.lib.orc_prefix(_p(pa, _f32p), pa.shape[0], _p(S, _f64p), _p(Q, _f64p))
        return S, Q

    def tstat(self, S, Q, w):
        n = S.shape[0] - 1
        t = np.empty(max(n, 1), dtype=np.float32)
        self.lib.orc_tstat(_p(S, _f64p), _p(Q, _f64p), n, w, _p(t, _f32p))
        return t[:n]

    def event_starts(self, raw, dig, off, rng, rna=0, thr_long=None):
        """event start positions of one read through the stage-level entry points, optionally with another
        threshold for the long detector (the reference's is 9.0 and its long detector hardly ever emits; tests lower
        it to exercise the code that handles long-detector peaks)"""
        pa = self.pa(raw, dig, off, rng)
        S, Q = self.prefix(pa)
        p = self.params(rna)
        t1, t2 = self.tstat(S, Q, p.w_short), self.tstat(S, Q, p.w_long)
        peaks = self.detect(t1, t2, rna, thr_long=thr_long)[0].astype(np.int64)
        n = len(raw)
        peaks = peaks[(peaks > 0) & (peaks < n)]
        return np.concatenate([np.zeros(1, np.int64), peaks]) if n else np.zeros(0, np.int64)

    def hot_lives(self, raw, dig, off, rng, rna=0, thr_long=None):
        """number of LIVES of the long detector (stretches between two resets by the short detector,
        events.c:414-422) that contain a stepped position with t2 > thr_long -- the only lives in which the long
        detector can emit (its peak_value must exceed the threshold, events.c:424). The detector is stepped one
        position at a time so that its masking can be observed. A walker that does not step the long detector must
        replay at least these lives."""
        pa = self.pa(raw, dig, off, rng)
        S, Q = self.prefix(pa)
        p = self.params(rna)
        if thr_long is not None:
            p.thr_long = float(thr_long)
        t1 = np.ascontiguousarray(self.tstat(S, Q, p.w_short), dtype=np.float32)
        t2 = np.ascontiguousarray(self.tstat(S, Q, p.w_long), dtype=np.float32)
        n = len(raw)
        s, l = self.Det(), self.Det()
        self.lib.orc_det_init(C.byref(s), C.byref(l))
        peaks = np.empty(4, dtype=np.uint64)
        lives, hot = 0, False
        for i in range(n):
            reset = s.peak_pos >= 0 and max(s.peak_value, float(t1[i])) > p.thr_short
            if reset:
                lives += int(hot)
                hot = False
            self.lib.orc_detect(_p(t1, _f32p), _p(t2, _f32p), i, i + 1, C.byref(p), C.byref(s), C.byref(l), _p(peaks, _u64p), 4)
            if l.masked_to < i and float(t2[i]) > p.thr_long:
                hot = True
        return lives + int(hot)

    def detect(self, t1, t2, rna, start=0, stop=None, cold=False, thr_long=None):
        """run the dual detector over [start, stop); -> (peaks, short_state, long_state)"""
        n = t1.shape[0]
        stop = n if stop is None else stop
        s, l = self.Det(), self.Det()
        if cold:
            self.lib.orc_det_cold(C.byref(s), C.byref(l), start)
        else:
            self.lib.orc_det_init(C.byref(s), C.byref(l))
        p = self.params(rna)
        if thr_long is not None:
            p.thr_long = float(thr_long)
        peaks = np.empty(max(n, 1), dtype=np.uint64)
        t1 = np.ascontiguousarray(t1, dtype=np.float32)
        t2 = np.ascontiguousarray(t2, dtype=np.float32)
        k = self.lib.orc_detect(_p(t1, _f32p), _p(t2, _f32p), start, stop, C.byref(p), C.byref(s), C.byref(l),
                                _p(peaks, _u64p), n)
        st = lambda d: (int(d.masked_to), int(d.peak_pos), float(d.peak_value), int(d.valid))
        return peaks[:k].copy(), st(s), st(l)


def have_ref() -> bool:
    return os.path.exists(REF_SO)


class Reference(_EventLib):
    """the unmodified reference functions (aborts on degenerate input, like the reference)"""

    def __init__(self):
        super().__init__(REF_SO, "ref_")

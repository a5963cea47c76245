"""Builds and loads tests/tools/jnn_set_oracle.c: the reference's jnn segmenter (jnn.c:176-282) with every field of
jnn_param_t general (sgpu_set_jnn), restated on the CPU sample by sample. TEST INFRASTRUCTURE ONLY.

JnnSetRef().jnn(raw, params) -> int64[k][2] (x, y) segments; .decrements(raw, params) -> how often the corrector
decremented err (jnn.c:213-217, 226-228) on that read. params: a (window, stall_len, error, seg_dist, corrector,
std_scale) tuple such as sigtk_b200.Jnn."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "tools", "jnn_set_oracle.c")

CDNA_R9 = (150, 0.25, 5, 50, 50, 0.75)   # JNNV1_CDNA_R9_PARAM (jnn.h:24-45), jnn_print's set when not rna
DRNA_R9 = (1000, 1.0, 5, 50, 50, 0.75)   # JNNV1_DRNA_R9_PARAM, jnn_print's set when rna
REFERENCE = {0: CDNA_R9, 1: DRNA_R9}


class Param(C.Structure):  # orc_jnn_param_t
    _fields_ = [("window", C.c_int32), ("stall_len", C.c_float), ("error", C.c_int32), ("seg_dist", C.c_int32),
                ("corrector", C.c_int32), ("std_scale", C.c_float)]


def _build() -> str:
    """the shared library next to the source, or in the temporary directory when tests/tools is read-only"""
    for d in (os.path.join(HERE, "tools"), tempfile.gettempdir()):
        out = os.path.join(d, "libjnnset.so")
        if os.path.exists(out) and os.path.getmtime(out) >= os.path.getmtime(SRC):
            return out
        if os.access(d, os.W_OK):
            tmp = out + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-std=c99", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", SRC,
                                   "-o", tmp, "-lm"])
            os.replace(tmp, out)
            return out
    raise RuntimeError("no writable directory for libjnnset.so")


class JnnSetRef:
    def __init__(self):
        self.lib = C.CDLL(_build())
        i16p, i64p = C.POINTER(C.c_int16), C.POINTER(C.c_int64)
        self.lib.orc_jnn_set.argtypes = [i16p, C.c_uint64, C.POINTER(Param), C.c_uint64, i64p]
        self.lib.orc_jnn_set.restype = C.c_int64
        self.lib.orc_jnn_set_counted.argtypes = [i16p, C.c_uint64, C.POINTER(Param), C.c_uint64, i64p, i64p]
        self.lib.orc_jnn_set_counted.restype = C.c_int64

    def _run(self, raw, params):
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        p = Param(int(params[0]), float(params[1]), int(params[2]), int(params[3]), int(params[4]), float(params[5]))
        cap = raw.shape[0] // 32 + 2
        xy = np.zeros(2 * cap, dtype=np.int64)
        n_dec = C.c_int64(0)
        k = self.lib.orc_jnn_set_counted(raw.ctypes.data_as(C.POINTER(C.c_int16)), raw.shape[0], C.byref(p), cap,
                                         xy.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(n_dec))
        assert k >= 0, k
        return xy[:2 * k].reshape(k, 2).copy(), int(n_dec.value)

    def jnn(self, raw, params):
        """segments of jnn_raw(raw, n, params) as int64[k][2]"""
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        p = Param(int(params[0]), float(params[1]), int(params[2]), int(params[3]), int(params[4]), float(params[5]))
        cap = raw.shape[0] // 32 + 2
        xy = np.zeros(2 * cap, dtype=np.int64)
        k = self.lib.orc_jnn_set(raw.ctypes.data_as(C.POINTER(C.c_int16)), raw.shape[0], C.byref(p), cap,
                                 xy.ctypes.data_as(C.POINTER(C.c_int64)))
        assert k >= 0, k
        return xy[:2 * k].reshape(k, 2).copy()

    def decrements(self, raw, params):
        """how often the corrector decremented err on this read"""
        return self._run(raw, params)[1]


def stall_reads(rng, n_reads, win, scale=1.0, outlier_every=2):
    """seeded int16 reads with stalls (flat stretches near the read's mean, of win/6 to 5 win samples), outliers
    inside them (every `outlier_every`-th read), gaps near and far from the merge distance, clipped spikes (every
    fifth read) and ragged lengths; -> [(raw, digitisation, offset, range)]"""
    out = []
    for k in range(n_reads):
        n = int(rng.integers(2 * win, int(40 * win * scale)))
        raw = (int(rng.integers(300, 700)) + rng.integers(20, 120) * rng.standard_normal(n)).astype(np.int64)
        pos = int(rng.integers(0, 2 * win))
        centre = int(np.mean(raw))
        while pos < n:
            stop = min(n, pos + int(rng.integers(max(win // 6, 1), 5 * win)))
            raw[pos:stop] = centre + rng.integers(-6, 7, stop - pos)
            if k % outlier_every == 1 and stop - pos > 60:
                raw[rng.integers(pos + 3, stop - 3, int(rng.integers(1, 60)))] = centre + 400
            pos = stop + int(rng.integers(3, 90) if k % 3 else rng.integers(30, 8 * win))
        if k % 5 == 0:
            raw[::911] = 9000
            raw[3::1777] = -900
        out.append((np.clip(raw, -32768, 32767).astype(np.int16), 8192.0, float(k % 7), 1400.0))
    return out


def random_set(rng, automaton):
    """a seeded jnn set sgpu_set_jnn accepts; automaton: error <= 6 < corrector, else error >= corrector"""
    while True:
        window = int(rng.integers(32, 1500))
        stall = float(np.float32(rng.uniform(0.03, 1.5)))
        if np.float32(window) * np.float32(stall) > 31:
            break
    seg_dist = int(rng.integers(-20, 400))
    scale = float(np.float32(rng.uniform(0.2, 1.6)))
    if automaton:
        error = int(rng.integers(0, 7))
        corrector = int(rng.integers(7, 300))
    else:
        corrector = int(rng.integers(0, 20))
        error = corrector + int(rng.integers(0, 40))
    return (window, stall, error, seg_dist, corrector, scale)

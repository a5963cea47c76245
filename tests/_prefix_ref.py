"""Builds and loads tests/tools/prefix_set_oracle.c: the reference's `sigtk prefix` (prefix_func, cfunc.c:169-234) with
every field of jnnv2's adaptor set and of find_polya's jnn_core set general (sgpu_set_prefix), restated on the CPU.
TEST INFRASTRUCTURE ONLY.

PrefixSetRef().prefix(raw, dig, off, rng, rna, p) -> (pos int64[4], stat float32[6]); .decrements(...) -> how often
the poly-A corrector decremented err (jnn.c:213-217, 226-228) on that read. p: a (adaptor, polya) pair of tuples such as
sigtk_b200.Prefix."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from sigtk_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "tools", "prefix_set_oracle.c")

RNA_R9 = (2000, 0.5, 1500, 2000, 200000)     # JNNV2_RNA_R9_ADAPTOR (jnn.h:88-102)
RNA004 = (2000, 0.7, 1500, 500, 200000)      # JNNV2_RNA_RNA004_ADAPTOR
POLYA_R9 = (250, 1.0, 30, 200, 50)           # JNNV1_R9_POLYA (jnn.h:47-56)
REFERENCE = {0: (RNA_R9, POLYA_R9), 1: (RNA004, POLYA_R9)}   # by SGPU_PARAM_PORE


class Adaptor(C.Structure):  # orc_adaptor_t
    _fields_ = [("window", C.c_int32), ("std_scale", C.c_float), ("seg_dist", C.c_int32), ("lo_thresh", C.c_int32),
                ("hi_thresh", C.c_int32)]


class Polya(C.Structure):  # orc_polya_t
    _fields_ = [("window", C.c_int32), ("stall_len", C.c_float), ("error", C.c_int32), ("seg_dist", C.c_int32),
                ("corrector", C.c_int32)]


def _build() -> str:
    """the shared library next to the source, or in the temporary directory when tests/tools is read-only"""
    for d in (os.path.join(HERE, "tools"), tempfile.gettempdir()):
        out = os.path.join(d, "libprefixset.so")
        if os.path.exists(out) and os.path.getmtime(out) >= os.path.getmtime(SRC):
            return out
        if os.access(d, os.W_OK):
            tmp = out + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-std=c99", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", SRC,
                                   "-o", tmp, "-lm"])
            os.replace(tmp, out)
            return out
    raise RuntimeError("no writable directory for libprefixset.so")


class PrefixSetRef:
    def __init__(self):
        self.lib = C.CDLL(_build())
        self.lib.orc_prefix_set.argtypes = [C.POINTER(C.c_int16), C.c_uint64, C.c_double, C.c_double, C.c_double,
                                            C.c_int, C.POINTER(Adaptor), C.POINTER(Polya), C.POINTER(C.c_int64),
                                            C.POINTER(C.c_float)]
        self.lib.orc_prefix_set.restype = C.c_int64

    def _run(self, raw, dig, off, rng, rna, p):
        raw = np.ascontiguousarray(raw, dtype=np.int16)
        a, y = p
        ca = Adaptor(int(a[0]), float(a[1]), int(a[2]), int(a[3]), int(a[4]))
        cy = Polya(int(y[0]), float(y[1]), int(y[2]), int(y[3]), int(y[4]))
        pos = np.zeros(4, dtype=np.int64)
        st = np.zeros(6, dtype=np.float32)
        n_dec = self.lib.orc_prefix_set(raw.ctypes.data_as(C.POINTER(C.c_int16)), raw.shape[0], dig, off, rng,
                                        int(rna), C.byref(ca), C.byref(cy), pos.ctypes.data_as(C.POINTER(C.c_int64)),
                                        st.ctypes.data_as(C.POINTER(C.c_float)))
        return pos, st, int(n_dec)

    def prefix(self, raw, dig, off, rng, rna, p):
        """prefix_func's numbers with the sets p = (adaptor, polya): (pos int64[4], stat float32[6])"""
        pos, st, _ = self._run(raw, dig, off, rng, rna, p)
        return pos, st

    def decrements(self, raw, dig, off, rng, rna, p):
        """how often the poly-A corrector decremented err on this read"""
        return self._run(raw, dig, off, rng, rna, p)[2]


def set_read(k, seed, p, n=None, polya=True):
    """a direct-RNA-like read shaped like test_gpu_prefix.adaptor_read, with the adaptor and poly-A stretches scaled to
    the sets p = (adaptor, polya): a low adaptor stretch long enough for a plausible run of the adaptor window, a
    poly-A plateau about 30 pA above it of a few poly-A windows (tolerated spikes inside when the set tolerates
    outliers), then the transcript. -> (raw, digitisation, offset, range)"""
    (aw, _, _, lo, hi), (pw, _, err, _, _) = p
    rng = np.random.default_rng([seed, k])
    a0 = int(rng.integers(max(aw // 4, 20), max(aw // 4, 20) + 2 * aw + 500))
    shortest = max(lo, 0) + aw + 50
    alen = int(rng.integers(shortest, shortest + max(2 * aw, 600)))
    if hi >= 0 and alen - aw > hi > 0:   # keep the run plausible where the set allows it
        alen = max(hi + aw - 50, aw + 20)
    pw = min(max(pw, 8), 3000)
    plen = int(rng.integers(pw + 30, pw * 8 + 300))
    if n is None:
        n = a0 + alen + plen + int(rng.integers(2000, 20000))
    rd = synth.make_read(k, n, seed=seed, p_change=0.025)
    raw = rd[0].astype(np.int32)
    scale = synth.DIGITISATION / synth.RANGE
    a1 = min(a0 + alen, n)
    lvl = 55.0 + 10.0 * rng.random()
    raw[a0:a1] = np.rint((lvl + rng.normal(0.0, 1.5, a1 - a0)) * scale - rd[2])
    if polya and a1 < n:
        p1 = min(a1 + plen, n)
        seg = np.rint((lvl + 30.0 + rng.normal(0.0, 2.5, p1 - a1)) * scale - rd[2])
        rate = 0.03 if err >= 30 else 0.002 if err > 0 else 0.0
        seg[rng.random(p1 - a1) < rate] += 400       # tolerated outliers inside the stretch
        raw[a1:p1] = seg
    return np.clip(raw, -32768, 32767).astype(np.int16), rd[1], rd[2], rd[3]


def random_set(rng, exact):
    """a seeded prefix set sgpu_set_prefix accepts; exact: polya error >= corrector, else error < corrector"""
    aw = int(rng.integers(2, 4000))
    adaptor = (aw, float(np.float32(rng.uniform(-0.3, 1.2))), int(rng.integers(-50, 3000)), int(rng.integers(1, 3000)),
               int(rng.integers(3000, 300000)))
    pw = int(rng.integers(-5, 600))
    stall = float(np.float32(rng.uniform(0.05, 2.0)))
    if exact:
        corrector = int(rng.integers(0, 40))
        error = corrector + int(rng.integers(0, 40))
    else:
        error = int(rng.integers(0, 80))
        corrector = error + int(rng.integers(1, 100))
    return adaptor, (pw, stall, error, int(rng.integers(-20, 400)), corrector)


# ---- the sets the tests use (shared by the CPU and GPU tests) ---------------------------------------------------------
INT32_MAX = 2**31 - 1
# custom adaptor sets, each with the reference's poly-A set
ADAPTORS = {
    "w4k": (2667, 0.6, 2000, 667, 266667),            # 2000 scaled from 3 kHz to 4 kHz (odd, 2667 % 8 = 3)
    "odd": (1501, 0.5, 1100, 1500, 150000),
    "lo_above_hi": (2000, 0.5, 1500, 5000, 100),      # no run is plausible
    "negative_merge": (1800, 0.5, -10, 1200, 200000),
    "negative_scale": (2000, -0.3, 1500, 2000, 200000),
    "smallest": (2, 0.5, 1500, 600, 200000),
    "largest": (13981, 0.5, 9000, 4000, 900000),
}
# poly-A sets on the automaton route (error < corrector), each with the R9 adaptor set
AUTOMATON = {
    "error0": (250, 1.0, 0, 200, 1),
    "error31": (250, 1.0, 31, 200, 50),
    "error32": (250, 1.0, 32, 200, 40),
    "error100": (250, 1.0, 100, 200, 150),
    "stall": (300, 0.4, 20, 100, 60),
    "window0": (0, 1.0, 10, 50, 40),
    "window_negative": (-5, 2.5, 10, -30, 40),
}
# poly-A sets on the exact route (error >= corrector: the corrector's decrement can act)
EXACT = {
    "corrector0": (100, 1.0, 5, 50, 0),
    "error_is_corrector": (250, 1.0, 30, 200, 30),
    "error_above": (150, 0.5, 40, 100, 10),
    "error_max": (250, 1.0, INT32_MAX, 200, 50),       # a stretch never closes
}


def named_set(name):
    """(adaptor, polya) of a set named in ADAPTORS, AUTOMATON or EXACT"""
    if name in ADAPTORS:
        return ADAPTORS[name], POLYA_R9
    return RNA_R9, AUTOMATON.get(name) or EXACT[name]


def without_corrector(p):
    """the same sets with a corrector that cannot act (corrector = error + 1): the result the automaton would give"""
    a, y = p
    return a, (y[0], y[1], y[2], y[3], min(y[2], INT32_MAX - 1) + 1)

"""A plain restatement of the statistics of `sigtk stat`, of the jnn band's moments and of the prefix statistics, written
from stat.h alone and independent of the C oracle; plus helpers that say where a float32 running sum changes binade,
meets a tie or stalls. TEST INFRASTRUCTURE ONLY.

meanf / stdvf (stat.h:17-44) add float32 values one after the other: here with np.add.accumulate, which is
sequential (np.sum is pairwise and would not do). pA is ((float)raw + (float)offset) * ((float)range / (float)dig)
(misc.c:15-32), the jnn signal the raw samples clamped to [0, 1200] (rm_outlier, jnn.c:58-75), a median the element
of rank n // 2 (ks_ksmall, stat.h:55-63)."""
from __future__ import annotations

import numpy as np

F = np.float32
SB, ROUND = 1024, 8192      # values per superblock, per round of the CTA role (8 warps)


def unit_of(dig, rng):
    with np.errstate(all="ignore"):
        return F(rng) / F(dig)


def pa(raw, dig, off, rng):
    with np.errstate(all="ignore"):
        return (np.asarray(raw).astype(F) + F(off)) * unit_of(dig, rng)


def clamp(raw):
    return np.clip(np.asarray(raw).astype(np.int32), 0, 1200).astype(F)


def running(x):
    """s[i] = fl(...fl(fl(x[0]) + x[1]) ... + x[i]) in float32"""
    with np.errstate(all="ignore"):
        return np.add.accumulate(np.asarray(x, F), dtype=F)


def meanf(x):
    x = np.asarray(x, F)
    with np.errstate(all="ignore"):
        return F(running(x)[-1]) / F(len(x))


def squares(x, m):
    with np.errstate(all="ignore"):
        d = np.asarray(x, F) - F(m)
        return d * d


def stdvf(x):
    x = np.asarray(x, F)
    with np.errstate(all="ignore"):
        return np.sqrt(F(running(squares(x, meanf(x)))[-1]) / F(len(x)))


def rank_half(x):
    return np.sort(np.asarray(x))[len(x) // 2]


def stat(raw, dig, off, rng):
    """the six numbers of stat_func (cfunc.c:126-159): mean, mean pA, stdv, stdv pA, median, median pA"""
    r, p = np.asarray(raw).astype(F), pa(raw, dig, off, rng)
    return np.array([meanf(r), meanf(p), stdvf(r), stdvf(p), rank_half(r), rank_half(p)], F)


def jnn_band(raw, std_scale=0.75):
    """(lo, hi) of jnn_core's band on the clamped signal: mean -/+ std_scale * stdv (jnn.c:181-185)"""
    c = clamp(raw)
    m, s = meanf(c), stdvf(c)
    b = s * F(std_scale)
    return m - b, m + b


def same_stat(a, b):
    """equal bit for bit, except that a NaN of either side only has to meet a NaN of the other"""
    a, b = np.asarray(a, F), np.asarray(b, F)
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32)))


# ---- where a running sum meets its edges -------------------------------------------------------------------------------
def exponent(s):
    """e with 2^e <= |s| < 2^(e+1) (s finite, nonzero)"""
    return np.frexp(np.asarray(s, np.float64))[1] - 1


def crossings(x):
    """positions i where the running sum of x (positive) enters a higher binade than s[i-1]'s"""
    s = running(x).astype(np.float64)
    prev = np.concatenate([[0.0], s[:-1]])
    ok = (prev > 0) & (s > 0) & np.isfinite(s)
    i = np.nonzero(ok)[0]
    return i[exponent(s[i]) > exponent(prev[i])]


def ties(x):
    """positions i > 0 where fl(s[i-1] + x[i]) was a tie: the exact sum lies halfway between two float32"""
    x = np.asarray(x, F)
    s = running(x)
    prev, xi = s[:-1].astype(np.float64), x[1:].astype(np.float64)
    exact = prev + xi                                   # exact: the operands are within 2^29 of each other here
    r = s[1:].astype(np.float64)
    with np.errstate(all="ignore"):
        other = np.where(exact > r, np.nextafter(s[1:], F(np.inf)), np.nextafter(s[1:], F(-np.inf))).astype(np.float64)
    mid = (exact != r) & (np.abs(exact - r) * 2 == np.abs(other - r))
    return np.nonzero(mid & np.isfinite(exact))[0] + 1


def stalls(x):
    """positions i > 0 where a nonzero x[i] left the running sum unchanged"""
    x = np.asarray(x, F)
    s = running(x)
    return np.nonzero((s[1:] == s[:-1]) & (x[1:] != 0))[0] + 1


def mantissa_after(x, first, last):
    """the running sum after x[last] as a multiple of the ulp of the sum before x[first] (its binade's mantissa
    integer S: 0xffffff is the binade's largest float, 0x1000000 its end)"""
    s = running(x).astype(np.float64)
    s0 = s[first - 1]
    ulp = 2.0 ** (exponent(s0) - 23)
    return s[last] / ulp


def where(i):
    """(round, warp, superblock, tile, lane) of position i of a read"""
    i = int(i)
    return i // ROUND, (i % ROUND) // SB, i // SB, (i % SB) // 32, i % 32

"""CPU checks of the exactness witness of the pA-input path (sigtk_b200/csrc/pa_input.cu), restated in numpy.

A read given as pA floats has its prefix sums formed by a parallel scan (tile sums, a scan of the tile sums within the
read, the samples of a tile on top) instead of the reference's sequential chain (events.c:293-303), but only when the
witness holds: all values finite, k = the smallest ulp exponent over the nonzero x (over the nonzero fl(x*x) for the
squares), sum |x| < 2^(k+53) and likewise for the squares. Then no FP64 addition rounds and any grouping gives the
reference's bits. Here the rule is checked against the oracle on adversarial arrays: where it holds, the tile-grouped
scan equals orc_prefix bit for bit and the events computed from it equal orc_getevents; arrays whose sums round fail
it, and some of them really do differ when summed in another order."""
import math

import numpy as np
import pytest

from _oracle import Oracle
from _oracle_pa import events_from_prefix, getevents_pa
from sigtk_b200 import synth

TILE = 4096   # samples per tile of pa_tile_kernel / pa_scan_kernel


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def ulp_exp(a):
    """ulp exponent of positive finite float32 values"""
    e = (np.asarray(a, np.float32).view(np.uint32) >> 23).astype(np.int64)
    return np.maximum(e, 1) - 150


def sum_exact(v):
    """sum |v| < 2^(k+53), k the smallest ulp exponent over the nonzero v (math.fsum rounds the exact sum to nearest,
    which keeps it on the same side of a power of two)"""
    nz = np.abs(v[v != 0])
    if nz.size == 0:
        return True
    return math.fsum(nz.astype(np.float64)) < 2.0 ** (int(ulp_exp(nz).min()) + 53)


def witness(x):
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        q = x * x                                   # float product (events.c:301)
    if not (np.all(np.isfinite(x)) and np.all(np.isfinite(q))):
        return False
    return sum_exact(x) and sum_exact(q)


def grouped_prefix(x):
    """S, Q (n+1 entries) the way the GPU groups the additions: tile sums, a scan of them, the tile's samples on top"""
    xd = np.asarray(x, np.float32).astype(np.float64)
    qd = (np.asarray(x, np.float32) * np.asarray(x, np.float32)).astype(np.float64)
    n = xd.shape[0]
    S, Q = np.zeros(n + 1), np.zeros(n + 1)
    cs = cq = 0.0
    for t0 in range(0, n, TILE):
        xs, qs = xd[t0:t0 + TILE], qd[t0:t0 + TILE]
        S[t0 + 1:t0 + 1 + xs.shape[0]] = cs + np.cumsum(xs)   # the tile's own running sums, then its offset
        Q[t0 + 1:t0 + 1 + qs.shape[0]] = cq + np.cumsum(qs)
        cs += float(np.sum(xs))          # (pairwise: another grouping again)
        cq += float(np.sum(qs))
    return S, Q


def events_from(orc, S, Q, rna):
    p = orc.params(rna)
    t1, t2 = orc.tstat(S, Q, p.w_short), orc.tstat(S, Q, p.w_long)
    return events_from_prefix(orc, orc.detect(t1, t2, rna)[0], S, Q)


def exact_arrays(orc):
    """arrays whose sums cannot round"""
    rng = np.random.default_rng(11)
    rd = synth.make_read(3, 30000, seed=11)
    out = {
        "pA of a synthetic read": orc.pa(*rd),
        "negated pA": -orc.pa(*rd),
        "integers in [-200, 200)": rng.integers(-200, 200, 20000).astype(np.float32),
        "zeros": np.zeros(9000, np.float32),
        "constant": np.full(10000, 87.25, np.float32),
        "subnormals and zeros": (rng.integers(-50, 50, 12000) * np.float32(2.0 ** -149)).astype(np.float32),
        "quarters near 2^10": (1024 + rng.integers(0, 64, 15000) / 4).astype(np.float32),
    }
    out["subnormals and zeros"][::3] = 0.0
    return out


def rounding_arrays():
    """arrays whose sums round in the reference's order"""
    rng = np.random.default_rng(12)
    sig = rng.normal(100.0, 15.0, 30000).astype(np.float32)
    med = np.median(sig)
    mad = np.median(np.abs(sig - med))
    wide = rng.normal(0.0, 1.0, 20000).astype(np.float32)
    wide[::997] = 3e7
    return {
        "(pA - median) / MAD": ((sig - med) / mad).astype(np.float32),
        "wide dynamic range": wide,
        "uniform (0, 1)": rng.random(20000).astype(np.float32),
    }


def test_witness_rule_on_small_cases():
    assert witness(np.zeros(0, np.float32)) and witness(np.zeros(5, np.float32))
    assert witness(np.array([1.0, 2.0, 3.0], np.float32))
    assert not witness(np.array([1.0, np.nan], np.float32))
    assert not witness(np.array([1.0, np.inf], np.float32))
    assert not witness(np.array([2e19, 1.0], np.float32))          # finite, but fl(x*x) overflows
    assert not witness(np.array([2.0 ** 30, 2.0 ** -24], np.float32))   # k = -47 (ulp of 2^-24): 2^30 > 2^6
    assert witness(np.array([2.0 ** 5, 1.0], np.float32))               # k = -23: 33 < 2^30, squares 1025 < 2^30
    assert not witness(np.array([2.0 ** 5, 2.0 ** -24], np.float32))    # x passes (32 < 2^6), the squares do not


@pytest.mark.parametrize("rna", [0, 1])
def test_witness_holds_and_any_grouping_is_exact(orc, rna):
    for name, x in exact_arrays(orc).items():
        assert witness(x), name
        S, Q = orc.prefix(x)
        gS, gQ = grouped_prefix(x)
        assert np.array_equal(S.view(np.uint64), gS.view(np.uint64)), name
        assert np.array_equal(Q.view(np.uint64), gQ.view(np.uint64)), name
        got = events_from(orc, gS, gQ, rna)
        want = getevents_pa(orc, x, rna)
        for a, b in zip(got, want):
            assert np.array_equal(np.asarray(a).view(np.uint32 if a.dtype == np.float32 else np.uint64),
                                  np.asarray(b).view(np.uint32 if b.dtype == np.float32 else np.uint64)), name


def test_witness_fails_where_sums_round(orc):
    differ = 0
    for name, x in rounding_arrays().items():
        assert not witness(x), name
        S, Q = orc.prefix(x)
        gS, gQ = grouped_prefix(x)
        differ += int(not (np.array_equal(S, gS) and np.array_equal(Q, gQ)))
    assert differ >= 1      # the order matters for these arrays: they must be summed in the reference's order

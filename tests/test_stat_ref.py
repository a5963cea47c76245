"""CPU tests that pin the plain statistics reference (tests/_stat_ref.py) and the crafted edge corpus
(tests/_stat_corpus.py) without a GPU: every crafted read really puts its edge (binade crossing, tie, stall, exact
mantissa end, negative or -0.0 addend, exponent at summable()'s limits) where its family says, and on every read the
plain reference gives the bits of orc_stat. The prefix reads find their adaptor (and, for RNA, their poly-A) under the
corpus's prefix set, at every residue mod 8 of the adaptor's start and length."""
import numpy as np
import pytest

import _stat_corpus as K
import _stat_ref as R
from _oracle import Oracle
from _prefix_ref import PrefixSetRef

CORPUS = K.corpus()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def test_running_sum_is_sequential():
    """np.add.accumulate adds float32 values one after the other (np.sum would add pairwise)"""
    rng = np.random.default_rng(1)
    for n in (1, 7, 1000, 5000):
        x = (rng.random(n) * 1000).astype(np.float32)
        s, want = np.float32(0), np.empty(n, np.float32)
        for i in range(n):
            s = np.float32(s + x[i])
            want[i] = s
        assert np.array_equal(R.running(x).view(np.uint32), want.view(np.uint32))
    x = np.full(1 << 18, 1000.5, np.float32)   # pairwise and sequential sums differ here
    assert R.running(x)[-1] != np.sum(x, dtype=np.float32)


@pytest.mark.parametrize("name,rd,check", CORPUS, ids=[c[0] for c in CORPUS])
def test_corpus_edges_and_oracle(orc, name, rd, check):
    check()
    assert R.same_stat(R.stat(*rd), orc.stat(*rd)), (name, R.stat(*rd), orc.stat(*rd))


def test_every_family_is_there():
    names = [c[0] for c in CORPUS]
    for fam in ("hit_", "ones_", "odd_ties", "jnn_1152", "cross_", "second_pass", "negative_", "minus_zero", "exp_",
                "unit_", "len_", "band_edges"):
        assert any(n.startswith(fam) for n in names), fam
    assert sorted(int(n[4:]) for n in names if n.startswith("len_")) == sorted(K.LENGTHS)


def test_median_reads(orc):
    for name, rd in K.median_reads():
        a = R.stat(*rd)
        assert R.same_stat(a, orc.stat(*rd)), name
        srt = np.sort(rd[0])
        n = len(srt)
        if name.startswith("edge_first"):
            assert (int(a[4]) + 32768) & 15 == 0 and srt[n // 2 - 1] != srt[n // 2]
        if name.startswith("edge_last"):
            assert (int(a[4]) + 32768) & 15 == 15 and srt[n // 2 + 1] != srt[n // 2]
    ns = sorted(int(n.split("_")[1]) for n, _ in K.median_reads() if n.startswith("tail_") and n.endswith("bin0"))
    assert ns == list(range(1, 18))


def test_degenerate_units(orc):
    """unit 0 and products that underflow to zero give pA of mixed +0 / -0: the oracle's median (qsort) and the plain
    reference's (np.sort) are zeros whose signs nothing pins; the GPU's is pA(raw median). The subnormal units are
    subnormal, and there every number agrees bit for bit."""
    for name, rd in K.degenerate_units():
        a, b = R.stat(*rd), orc.stat(*rd)
        u = R.unit_of(rd[1], rd[3])
        if K.mixed_zero(name):
            z = R.pa(*rd)
            z = z[z == 0]
            assert np.signbit(z).any() and (~np.signbit(z)).any(), name
            assert a[5] == 0 and b[5] == 0, name
            assert R.same_stat(a[:5], b[:5]), name
        else:
            assert 0 < abs(float(u)) < 2.0 ** -126, (name, u)
            assert R.same_stat(a, b), name


def test_prefix_reads_place_their_stretches():
    ref = PrefixSetRef()
    for sign in (1.0, -1.0):
        for rna in (0, 1):
            ax, ln, px, polya, flips = set(), set(), set(), 0, 0
            for rd in K.prefix_reads(sign):
                pos, st = ref.prefix(*rd, rna, K.PREFIX_SET)
                assert pos[1] > 0, pos
                ax.add(int(pos[0]) % 8)
                ln.add(int(pos[1] - pos[0]) % 8)
                p = R.pa(*rd)[pos[0]:pos[1]]
                assert R.same_stat([R.meanf(p), R.stdvf(p), R.rank_half(p)], st[:3])
                srt = np.sort(rd[0][pos[0]:pos[1]])
                flips += len(srt) % 2 == 0 and srt[len(srt) // 2] != srt[len(srt) // 2 - 1]
                if pos[3] > 0:
                    polya += 1
                    px.add(int(pos[1] + pos[2]) % 8)
                    srt = np.sort(rd[0][pos[1] + pos[2]:pos[1] + pos[3]])
                    flips += len(srt) % 2 == 0 and srt[len(srt) // 2] != srt[len(srt) // 2 - 1]
                    q = R.pa(*rd)[pos[1] + pos[2]:pos[1] + pos[3]]
                    assert R.same_stat([R.meanf(q), R.stdvf(q), R.rank_half(q)], st[3:])
            assert ax == set(range(8)) and ln == set(range(8)), (ax, ln)
            assert flips >= 4   # even stretches whose two middle samples differ: the rank from the other end matters
            if rna and sign > 0:
                assert polya == len(K.prefix_reads()) and px == set(range(8)), (polya, px)


def test_long_prefix_stretches_are_summarised():
    """the long adaptors span several superblocks of range_moments, and their pA sum is exactly 2^14 at the end of
    the stretch's superblock 1"""
    ref = PrefixSetRef()
    for sign in (1.0, -1.0):
        for rd in K.long_prefix_reads(sign):
            pos, _ = ref.prefix(*rd, 1, K.PREFIX_SET)
            assert pos[1] - pos[0] > 4 * R.SB, pos
            p = R.pa(*rd)[pos[0]:pos[1]]
            assert abs(float(R.running(p)[2 * R.SB - 1])) == 2.0 ** 14
            assert R.mantissa_after(np.abs(p), R.SB + 31 * 32, 2 * R.SB - 1) == 0x1000000

"""Crafted reads that put the edges of the ordered float sums (float_order.cuh, stat.cu, prefix.cu) and of the median
select where they are wanted, each with the check that the edge really is there. TEST INFRASTRUCTURE ONLY.

A case is (name, (raw, dig, off, rng), check); check() asserts, through the plain reference's helpers, that the
case's binade crossings, ties, stalls or exact mantissa ends fall at the intended (round, warp, superblock, tile,
lane). Positions: a superblock is 1,024 values (32 tiles of 32, one lane per value of a tile in the summary), a round
of the one-CTA-per-read role is 8 superblocks (one per warp). The calibration is the ordinary (digitisation, offset,
range) triple: range = 2^k, digitisation = 1 gives the power-of-two unit 2^k."""
from __future__ import annotations

import numpy as np

import _stat_ref as R

F = np.float32
TWO24 = 1 << 24
LONG = 2_000_000


def hit(target, at):
    """at + 1 non-negative integers (int16 range) whose running sum is exactly `target` after the last one"""
    base, rem = divmod(int(target), at + 1)
    assert base + 1 <= 32767, (target, at)
    v = np.full(at + 1, base, np.int64)
    v[:rem] += 1
    return v


def i16(v):
    v = np.asarray(v, np.int64)
    assert v.min() >= -32768 and v.max() <= 32767
    return v.astype(np.int16)


def pos(sb, tile=31, lane=31):
    return sb * R.SB + tile * 32 + lane


def channels(rd):
    raw, dig, off, rng = rd
    return raw.astype(F), R.pa(raw, dig, off, rng)


def second_pass(x):
    return R.squares(x, R.meanf(x))


def expect(cond, what):
    assert cond, what


# ---- the families --------------------------------------------------------------------------------------------------------
def exact_hits():
    """the running raw sum (and the pA sum: pA = raw / 8) is exactly 2^24 - 1 or 2^24 after the last value of a tile
    in the middle of a superblock, of a superblock, of a round; and exactly 2^24 at a tile end inside a round where
    the sum then goes on (the mantissa integer of the tile's binade reaches 0xffffff, or 0x1000000: the binade ends
    on the tile's last value)"""
    out = []
    for tgt in (TWO24 - 1, TWO24):
        for where_, p in (("tile", pos(8 + 2, 12)), ("superblock", pos(8 + 5)), ("round", pos(15))):
            v = np.concatenate([hit(tgt, p), np.tile([2, 4, 6, 2], 1500)])
            rd = (i16(v), 1.0, 0.0, 0.125)

            def check(rd=rd, p=p, tgt=tgt):
                for x in channels(rd):
                    s = R.running(x).astype(np.float64)
                    expect(s[p] == tgt * float(x[0] / rd[0][0]), f"sum {s[p]} at {p}")
                    S = R.mantissa_after(x, p - 31, p)
                    expect(S == (0xFFFFFF if tgt < TWO24 else 0x1000000), f"mantissa {S}")
            out.append((f"hit_{tgt:#x}_{where_}", rd, check))
    return out


def ones():
    """(a) ones: the sums are 2^k exactly at the end of superblocks and of rounds (0x1000000 at the end of a summary);
    pA = 2: at other superblock ends. (b) a head that brings the sum to 2^24 - 1024 in the first superblock, then
    ones: 2^24 exactly at the end of superblock 1, after that every one is a tie and the sum stalls at 16,777,216
    for 2,000,000 samples (the mean is 2^24 / n)."""
    a = (np.ones(300_000, np.int16), 1.0, 1.0, 1.0)

    def check_a(rd=a):
        r, p = channels(rd)
        cr, cp = R.crossings(r), R.crossings(p)
        for k in (11, 13, 14, 17):
            expect((1 << k) - 1 in cr, f"raw 2^{k}")
            expect((1 << (k - 1)) - 1 in cp, f"pA 2^{k}")
        expect(R.where(8191)[:2] == (0, 7) and R.where(16383)[:2] == (1, 7), "round ends")

    head = np.full(R.SB, (TWO24 - R.SB) // R.SB, np.int64)
    b = (i16(np.concatenate([head, np.ones(LONG - R.SB, np.int64)])), 1.0, 0.0, 1.0)

    def check_b(rd=b):
        for x in channels(rd):
            s = R.running(x)
            expect(float(s[2047]) == TWO24 and float(s[2046]) < TWO24, "2^24 at the end of superblock 1")
            st = R.stalls(x)
            expect(len(st) == LONG - 2048 and st[0] == 2048, "stalls from 2048 on")
            t = R.ties(x)
            expect(len(t) == LONG - 2048 and t[0] == 2048, "a tie at every step from 2048 on")
    return [("ones_300k", a, check_a), ("ones_stall_2M", b, check_b)]


def ties_everywhere():
    """(a) the sum at 2^24 after the first superblock, then odd integers: every step a tie (ulp 2), rounded up or
    down by the parity of the mantissa; pA = raw / 1024 ties the same way. (b) 1152 everywhere (the jnn clamp keeps
    it): past 2^31 (ulp 256) every step adds 4.5 ulp, a tie; 2,000,000 samples."""
    head = np.full(R.SB, TWO24 // R.SB, np.int64)
    body = np.tile([3, 5, 7, 1, 9, 11, 3, 1], 5000)
    a = (i16(np.concatenate([head, body])), 1.0, 0.0, 1.0 / 1024)

    def check_a(rd=a):
        for x in channels(rd):
            t = R.ties(x)
            expect(np.array_equal(t, np.arange(R.SB, len(x))), "a tie at every step after the head")
    b = (np.full(LONG, 1152, np.int16), 1.0, 0.0, 1.0)

    def check_b(rd=b):
        x = R.clamp(rd[0])
        s = R.running(x)
        first = int(np.argmax(s.astype(np.float64) >= 2.0 ** 31))
        t = R.ties(x)
        expect(first > 0 and len(t) >= LONG - first - 1 and t[-1] == LONG - 1, "ties past 2^31")
    return [("odd_ties", a, check_a), ("jnn_1152_2M", b, check_b)]


def crossings_placed():
    """binade crossings placed: in the first tile of superblock 2, in the last tile of superblock 3, in the partial last
    tile of a read; the raw and the pA sum (pA = raw - 21) crossing 2^19 and 2^20 at different warps of the same
    round; second-pass crossings: m -/+ d alternating (the mean is m exactly, every square d^2), so the squares' sum is
    2^k exactly at superblock and round ends (d = 16), or crosses inside tiles (d = 17)"""
    out = []
    for name, v, n, k, want in (("first_tile", 127, 5000, 18, (2, 0)), ("last_tile", 257, 6000, 20, (3, 31)),
                                ("partial_last_tile", 257, 4085, 20, (3, 31))):
        rd = (np.full(n, v, np.int16), 1.0, 0.0, 1.0)

        def check(rd=rd, k=k, want=want):
            for x in channels(rd):
                c = [i for i in R.crossings(x) if R.running(x)[i] >= 2.0 ** k][0]
                expect(R.where(c)[2:4] == want, f"crossing of 2^{k} at {R.where(c)}")
        out.append((f"cross_{name}", rd, check))
    two = (np.full(20000, 97, np.int16), 1.0, -21.0, 1.0)

    def check_two(rd=two):
        r, p = channels(rd)
        for k, rnd, wr, wp in ((19, 0, 5, 6), (20, 1, 2, 5)):
            cr = [i for i in R.crossings(r) if R.running(r)[i] >= 2.0 ** k][0]
            cp = [i for i in R.crossings(p) if R.running(p)[i] >= 2.0 ** k][0]
            expect(R.where(cr)[:2] == (rnd, wr) and R.where(cp)[:2] == (rnd, wp), (R.where(cr), R.where(cp)))
    out.append(("cross_two_channels", two, check_two))
    for d in (16, 17):
        rd = (i16(400 + d * np.tile([1, -1], 20000)), 1.0, 0.0, 1.0)

        def check_sq(rd=rd, d=d):
            for x in channels(rd):
                expect(R.meanf(x) == 400, "mean exact")
                q = second_pass(x)
                c = R.crossings(q)
                if d == 16:
                    expect(all(((1 << (k - 8)) - 1) in c for k in range(18, 24)), "exact second-pass ends")
                    expect(R.mantissa_after(q, 8191 - 31, 8191) == 0x1000000, "round end")
                else:
                    expect(any(R.where(i)[3:] != (31, 31) and R.where(i)[4] not in (0, 31) for i in c), "inside")
        out.append((f"second_pass_d{d}", rd, check_sq))
    return out


def unsummarisable():
    """tiles that cannot be summarised among ones that can. (a) raw: the sum in [2^24, 2^25) (ulp 2), then 2s, and
    whole tiles of -9, +10 (-4.5 ulp: a tie, then +5 ulp) as the first, a middle or the last tile of a superblock
    and of a round; pA = raw / 4 the same. (b) pA of both signs with a positive pA sum (unit 1, offset -3): raw
    values 2 give pA -1 in the first tile of superblock 1, in the middle and last tile of others. (c) -0.0 pA: unit
    -1, offset 100, raw = -100 in the first, a middle and the last tile; every other pA is positive."""
    head = np.concatenate([np.full(R.SB, TWO24 // R.SB, np.int64), np.full(256, 32767, np.int64)])
    n = 20000
    v = np.concatenate([head, np.full(n - len(head), 2, np.int64)])
    bad_tiles = [(3, 0), (5, 13), (7, 31), (8, 0), (12, 31), (15, 0), (16, 13)]
    for sb, t in bad_tiles:
        v[pos(sb, t, 0): pos(sb, t, 0) + 32] = np.tile([-9, 10], 16)
    a = (i16(v), 1.0, 0.0, 0.25)

    def check_a(rd=a):
        for x in channels(rd):
            s = R.running(x)
            expect(bool((s[1:] > 0).all()) and float(s[-1]) < 2.0 ** 25, "positive, below 2^25")
            t = set(R.ties(x).tolist())
            for sb, tl in bad_tiles:
                expect(pos(sb, tl, 0) in t, f"tie in tile {sb}/{tl}")
    bv = np.full(12000, 40, np.int64)
    places = [(1, 0, 0), (2, 13, 7), (3, 31, 31), (8, 0, 5), (9, 31, 0)]
    for sb, t, l in places:
        bv[pos(sb, t, l)] = 2
    b = (i16(bv), 1.0, -3.0, 1.0)

    def check_b(rd=b):
        p = R.pa(*rd)
        expect(all(p[pos(*q)] == -1 for q in places) and (R.running(p) > 0).all(), "negative pA, positive sum")
    cv = np.full(12000, -140, np.int64)
    for sb, t, l in places:
        cv[pos(sb, t, l)] = -100
    c = (i16(cv), 1.0, 100.0, -1.0)

    def check_c(rd=c):
        p = R.pa(*rd)
        z = [pos(*q) for q in places]
        expect(all(p[i] == 0 and np.signbit(p[i]) for i in z) and (p[np.setdiff1d(np.arange(len(p)), z)] > 0).all(),
               "-0.0 pA")
    return [("negative_tiles", a, check_a), ("negative_pa", b, check_b), ("minus_zero_pa", c, check_c)]


def exponents():
    """accumulators at summable()'s limits: pA = 300 * 2^-119 over 6,000 samples (exponents -111 .. -99), 300 * 2^80
    over 12,000 (88 .. 101); second pass: m -/+ 16 with units 2^-57 and 2^45 (squares 2^-106 and 2^98 per step, the
    sums through exponents -101 .. -99 and 99 .. 101); unit +inf, -inf (digitisation 0) and NaN (0 / 0)"""
    out = []
    for name, raw, k, pas in (("tiny", np.full(6000, 300, np.int16), -119, 1),
                              ("huge", np.full(12000, 300, np.int16), 80, 1),
                              ("tiny_sq", i16(400 + 16 * np.tile([1, -1], 20000)), -57, 2),
                              ("huge_sq", i16(400 + 16 * np.tile([1, -1], 20000)), 45, 2)):
        rd = (raw, 1.0, 0.0, 2.0 ** k)

        def check(rd=rd, pas=pas):
            p = R.pa(*rd)
            x = p if pas == 1 else second_pass(p)
            e = set(R.exponent(R.running(x)).tolist())
            lim = (-101, -100, -99) if rd[3] < 1 else (99, 100, 101)
            expect(all(q in e for q in lim), f"exponents {sorted(e)[:3]}..{sorted(e)[-3:]}")
        out.append((f"exp_{name}", rd, check))
    sig = (np.arange(5000) * 7919 % 1400 + 100).astype(np.int16)
    for name, dig, rng in (("inf", 0.0, 1402.882324), ("minus_inf", 0.0, -1402.882324), ("nan", 0.0, 0.0)):
        rd = (sig, dig, 0.5, rng)

        def check(rd=rd, name=name):
            u = R.unit_of(rd[1], rd[3])
            expect(np.isnan(u) if name == "nan" else np.isinf(u), "unit")
        out.append((f"unit_{name}", rd, check))
    return out


LENGTHS = (1, 2, 31, 32, 33, 1023, 1024, 1025, 8191, 8192, 8193, 131071, 131072, 131073)


def lengths():
    """the role and block sizes: a periodic signal whose sums cross binades and meet ties (pA = (raw - 3.5) / 2)"""
    base = (np.arange(max(LENGTHS)) * 7919 % 997 + 200).astype(np.int16)
    out = []
    for n in LENGTHS:
        rd = (base[:n].copy(), 1.0, -3.5, 0.5)

        def check(rd=rd):
            x = channels(rd)[1]
            expect(len(x) < 20000 or len(R.ties(x)) > 0, "ties")
        out.append((f"len_{n}", rd, check))
    return out


def jnn_segments(raw, std_scale):
    """`sigtk jnn`'s DNA segmenter (JNNV1_CDNA_R9_PARAM) with another std_scale: the band mean -/+ std_scale * stdv"""
    from _jnn_ref import CDNA_R9, JnnSetRef
    global _JNN
    if "_JNN" not in globals():
        _JNN = JnnSetRef()
    return _JNN.jnn(raw, CDNA_R9[:5] + (std_scale,))


WIDER, NARROWER = float(F(0.75) + F(2.0 ** -18)), float(F(0.75) - F(2.0 ** -18))   # the band +/- one ulp at 588, 612


def band_edges():
    """jnn bands that end on samples or one ulp past them. Levels 600 -/+ 16 (n0 each), -/+ 12 (9 m each), -/+ 20
    (7 m each) give a mean of 600 and a stdv of 16 exactly, so the band (600 -/+ 0.75 * 16) ends exactly on the
    samples 588 and 612 ("on"): they are outside it, and a band one ulp wider (std_scale 0.75 + 2^-18) takes them in.
    Four more pairs 600 -/+ 17 and one 600 raise the stdv just enough that the band ends one ulp past 588 and 612
    ("past"): they are inside it, and a band one ulp narrower leaves them out. The 588s and the 612s come in runs of
    at least 150 samples (the DNA window), so either change of the band changes the segments."""
    out = []
    for k, (n0, m) in enumerate(((400, 40), (1000, 100), (300, 60))):
        for kind in ("on", "past"):
            rng = np.random.default_rng(k)
            extra = [617] * 4 + [583] * 4 + [600] if kind == "past" else []
            outer = np.array([584] * n0 + [616] * n0 + [580] * 7 * m + [620] * 7 * m + extra)
            rng.shuffle(outer)
            h = 9 * m // 2
            runs = [np.full(h, 588), np.full(h, 612), np.full(9 * m - h, 588), np.full(9 * m - h, 612)]
            chunks = np.array_split(outer, 5)
            raw = np.concatenate([chunks[0]] + [x for pair in zip(runs, chunks[1:]) for x in pair])
            rd = (i16(raw), 1.0, 0.0, 1.0)

            def check(rd=rd, kind=kind):
                lo, hi = R.jnn_band(rd[0])
                want = (588.0, 612.0) if kind == "on" else (float(np.nextafter(F(588), F(0))),
                                                            float(np.nextafter(F(612), F(1e9))))
                expect((float(lo), float(hi)) == want, (lo, hi))
                seg = jnn_segments(rd[0], 0.75)
                moved = jnn_segments(rd[0], WIDER if kind == "on" else NARROWER)
                expect(not np.array_equal(seg, moved), "a band one ulp off gives other segments")
            out.append((f"band_edges_{kind}_{k}", rd, check))
    return out


def corpus():
    return (exact_hits() + ones() + ties_everywhere() + crossings_placed() + unsummarisable() + exponents() + lengths()
            + band_edges())


# ---- medians -------------------------------------------------------------------------------------------------------------
def median_reads():
    """the select at its bin edges: one bin of 16 values; rank n // 2 on the first key of a bin (key & 15 == 0) and on
    the last (15); keys -32768 and 32767; two-valued reads with rank n // 2 exactly on the boundary; n = 1 .. 17 (every
    tail of a 128-bit word) with values in the bin of 0 (a zero sample past the read is in the median's bin) and in the
    bin above it (a zero past the read is below the median); unit < 0"""
    rng = np.random.default_rng(5)
    out = []
    out.append(("one_bin", (i16(592 + rng.integers(0, 16, 1001)), 8192.0, 3.0, 1402.882324)))
    for n in (100, 101):
        h = n // 2
        out.append((f"edge_first_{n}", (i16([591] * h + [592] * (n - h)), 8192.0, 3.0, 1402.882324)))
        out.append((f"edge_last_{n}", (i16([591] * (h + 1) + [592] * (n - h - 1)), 8192.0, 3.0, 1402.882324)))
        out.append((f"min_key_{n}", (i16([-32768] * (h + 1) + [-32767] * (n - h - 1)), 8192.0, 0.0, 1402.882324)))
        out.append((f"max_key_{n}", (i16([32766] * h + [32767] * (n - h)), 8192.0, 0.0, 1402.882324)))
        out.append((f"negative_unit_{n}", (i16(rng.permutation([607] * h + [608] * (n - h))), 8192.0, 3.0, -1402.882324)))
    for n in range(1, 18):
        out.append((f"tail_{n}_bin0", (i16(rng.integers(0, 16, n)), 8192.0, 3.0, 1402.882324)))
        out.append((f"tail_{n}_bin1", (i16(rng.integers(16, 32, n)), 8192.0, 3.0, 1402.882324)))
        out.append((f"tail_{n}_edge", (i16(rng.permutation([15] * (n // 2) + [16] * (n - n // 2))), 8192.0, 3.0,
                                       -1402.882324)))
    out.append(("long_edge", (i16(rng.permutation([1023] * 100000 + [1024] * 100001)), 8192.0, 3.0, 1402.882324)))
    return out


def degenerate_units():
    """calibrations at the bottom of float: (a) unit 0 (range 0) and (b) unit 2^-149 with offset 0.5, where raw 0 and
    -1 give +/-0.5 * 2^-149, which rounds to +0 and -0: pA of mixed +0 / -0, the samples in order and shuffled, the
    median's raw sample negative in some, positive in others; (c) subnormal units (range 2^-140 over digitisation 1,
    range 2^-100 over 2^30, and negative): every pA a nonzero subnormal but the one of raw == -offset, exact in
    every number, the moments added value by value (summable() refuses exponent field 0)"""
    rng = np.random.default_rng(9)
    out = []
    for k, raw in enumerate((np.arange(-60, 41), np.arange(-40, 61), rng.permutation(np.arange(-60, 41)),
                             rng.permutation(np.arange(-50, 52)))):
        out.append((f"unit_zero_{k}", (i16(raw), 8192.0, 0.0, 0.0)))
        out.append((f"underflow_{k}", (i16(np.clip(raw, -1, 0) if k % 2 else np.where(raw < 0, -1, raw)), 1.0, 0.5,
                                       2.0 ** -149)))
    for k, (dig, rng_) in enumerate(((1.0, 2.0 ** -140), (2.0 ** 30, 2.0 ** -100), (1.0, -(2.0 ** -140)))):
        out.append((f"subnormal_{k}", (i16(rng.permutation(np.arange(-60, 41)) * (1 + 20 * k)), dig, 0.0, rng_)))
        out.append((f"subnormal_frac_{k}", (i16(rng.integers(-300, 300, 1500)), dig, 0.25, rng_)))
    return out


def mixed_zero(name):
    """a degenerate read whose pA median is a zero of a sign nothing pins"""
    return name.startswith(("unit_zero", "underflow"))


# ---- prefix reads ----------------------------------------------------------------------------------------------------------
PREFIX_SET = ((16, 1.0, 8, 50, 100000), (40, 1.0, 3, 20, 50))   # window 16 adaptor set; poly-A automaton (3 < 50)


def prefix_reads(unit_sign=1.0):
    """reads for PREFIX_SET: 1100 before and after, an adaptor of 191s then 192s and a poly-A of 671s then 672s (pA =
    raw / 16: in the band (adaptor mean + 30) -/+ 20); the adaptor's start, its length and the poly-A's length chosen
    so that the adaptor's start and length and the poly-A's start take every residue mod 8. The set finds the adaptor at
    [a0 + 1, a1 + 3) and the poly-A at [a1 + 3, p1) of the step positions a0, a1, p1; the steps from 191 to 192 and
    from 671 to 672 are placed so that in a stretch of even length the two middle samples are 191 and 192 (671 and
    672): its median sits on a bin edge (192 and 672 are multiples of 16) and a negative unit takes the other one."""
    out = []
    for k in range(32):
        a0, alen, plen = 300 + k % 8, 400 + 3 * (k % 8) + k // 8, 300 + 5 * k
        la, lp = alen + 2, plen - 3
        ad = np.where(np.arange(alen) < 1 + la // 2, 191, 192)
        po = np.where(np.arange(plen) < 3 + lp // 2, 671, 672)
        v = np.concatenate([np.full(a0, 1100), ad, po, np.full(1500 + 13 * k, 1100)])
        out.append((i16(v), 1.0, 0.0, unit_sign / 16.0))
    return out + long_prefix_reads(unit_sign)


def long_prefix_reads(unit_sign=1.0):
    """adaptors of more than 4,096 samples, so that range_moments sums them over several superblocks: the set finds
    the adaptor at [a0 + 4, a1 - 3) of its step positions and the poly-A at [a1, p1). The adaptor's first 2,048
    samples are 128 (pA 8): its pA sum is exactly 2^14 at the end of its superblock 1 (the mantissa integer reaches
    0x1000000 on a summarised superblock); then 127s, as many as half the stretch, then 128s again, so that
    the median sits on the bin edge 127 / 128 and a negative unit takes the other middle sample."""
    out = []
    for k in range(4):
        a0, alen, plen = 300 + 3 * k, 4300 + 5 * k, 400 + k
        la = alen - 7
        ad = np.full(alen, 128)
        ad[4 + 2048: 4 + 2048 + la // 2] = 127
        po = np.where(np.arange(plen) < plen // 2, 671, 672)
        v = np.concatenate([np.full(a0, 1100), ad, po, np.full(9000, 1100)])
        out.append((i16(v), 1.0, 0.0, unit_sign / 16.0))
    return out

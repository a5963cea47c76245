"""CPU checks of the caller's own jnn parameters (sgpu_set_jnn) -- test infrastructure and the reformulation the
kernels rest on, no GPU:

  - orc_jnn_set (tests/tools/jnn_set_oracle.c, every field of jnn_param_t general) with jnn_print's two sets equals
    the compiled reference's stored stdout and the oracle's orc_jnn;
  - jnn_walk_kernel's data flow (an automaton of error + 2 states over the in-band bit, word maps composed by a prefix
    scan, at most one candidate per word), restated in Python with a set's window / first_min / seg_dist / std_scale
    and CLOSED = error + 1, equals orc_jnn_set for seeded sets with error <= 6 < corrector;
  - the corrector's decrement never fires when error < corrector, and does fire, changing the segments, for a set with
    error >= corrector: the case jnn_exact_kernel exists for."""
import math
import os

import numpy as np
import pytest

import _fmt
from _jnn_ref import CDNA_R9, DRNA_R9, REFERENCE, JnnSetRef, random_set, stall_reads
from _oracle import Oracle

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INT32_MAX = 2 ** 31 - 1


@pytest.fixture(scope="module")
def ref():
    return JnnSetRef()


# ---- the automaton of jnn_walk_kernel, for any set with error <= 6 < corrector ---------------------------------------
def _ffs(x):
    return (x & -x).bit_length()


def _clz(x):
    return 32 - x.bit_length()


def _popc(x):
    return bin(x).count("1")


def word_end(bits, zeros, m, s, closed):
    """jnn_word_end: state after the m samples of a word entered in state s"""
    j = 0
    while j < m:
        if s == closed:
            rest = bits >> j
            if rest == 0:
                return closed
            j += _ffs(rest) - 1
            s = 0
        z = zeros >> j
        need = closed - s
        nz = _popc(z)
        if nz < need:
            return s + nz
        for _ in range(1, need):
            z &= z - 1
        j += _ffs(z)
        s = closed
    return s


def band_of(raw, std_scale):
    """mean -/+ fl(stdv * std_scale) of the clamped signal, float32 sums in sample order (jnn.c:181-185), as the
    integers just inside it (jnn_band)"""
    sig = np.clip(raw, 0, 1200).astype(np.float32)
    acc = np.float32(0)
    for v in sig:
        acc = np.float32(acc + v)
    mn = np.float32(acc / np.float32(len(sig)))
    dev = np.float32(0)
    for v in sig:
        d = np.float32(v - mn)
        dev = np.float32(dev + np.float32(d * d))
    sd = np.float32(np.sqrt(np.float32(dev / np.float32(len(sig)))))
    band = np.float32(sd * np.float32(std_scale))
    top, bot = np.float32(mn + band), np.float32(mn - band)
    hi_i = int(math.ceil(min(max(float(top), -1.0), 2000.0))) - 1
    lo_i = int(math.floor(min(max(float(bot), -2.0), 2000.0))) + 1
    return lo_i, hi_i


def walk(raw, params):
    """jnn_walk_kernel's data flow for one read (carries between 1024-sample blocks: state, opening position,
    previous word)"""
    window, stall, error, seg_dist, corrector, std_scale = params
    assert 0 <= error <= 6 and error < corrector
    closed = error + 1
    n = len(raw)
    if n == 0:
        return np.zeros((0, 2), np.int64)
    lo_i, hi_i = band_of(raw, std_scale)
    first_min = np.float32(window) * np.float32(stall)
    cand_min = min(np.float32(window), first_min)
    sv = np.clip(raw.astype(np.int64), 0, 1200)
    inb = (sv >= lo_i) & (sv <= hi_i)
    n_seg = last_y = 0
    out = []
    state, open_pos, last_word = closed, 0, 0xFFFFFFFF
    for t0 in range(0, n, 1024):
        ins, zs, ms, maps = [], [], [], []
        for lane in range(32):
            i0 = t0 + lane * 32
            m = max(0, min(32, n - i0))
            bits = int((inb[i0:i0 + m].astype(np.uint64) << np.arange(m, dtype=np.uint64)).sum()) if m > 0 else 0
            valid = 0xFFFFFFFF if m == 32 else (1 << m) - 1
            ins.append(bits)
            zs.append(~bits & valid)
            ms.append(m)
            maps.append([word_end(bits, zs[-1], m, s, closed) for s in range(closed + 1)])
        s_in, cur = [], state
        for lane in range(32):  # the prefix scan of the maps
            s_in.append(cur)
            cur = maps[lane][cur]
        close, perr, last_open = [-1] * 32, [0] * 32, [-1] * 32
        for lane in range(32):
            i0, bits, zeros, m = t0 + lane * 32, ins[lane], zs[lane], ms[lane]
            prev_in = ins[lane - 1] if lane else last_word
            j, s = 0, s_in[lane]
            while j < m:
                if s == closed:
                    rest = bits >> j
                    if rest == 0:
                        break
                    j += _ffs(rest) - 1
                    s = 0
                    last_open[lane] = i0 + j
                z = zeros >> j
                need = closed - s
                if _popc(z) < need:
                    break
                for _ in range(1, need):
                    z &= z - 1
                pos = j + _ffs(z) - 1
                if j == 0 and s_in[lane] != closed and close[lane] < 0:
                    close[lane] = pos
                    below = (bits & ((1 << pos) - 1)) if pos else 0
                    perr[lane] = (pos - 1) - (31 - _clz(below)) if below else pos + _clz(prev_in)
                j, s = pos + 1, closed
        run = open_pos
        for lane in range(32):
            if close[lane] >= 0:
                i0 = t0 + lane * 32
                c, en = i0 + close[lane] - run, i0 + close[lane] - perr[lane]
                if np.float32(c) >= cand_min and (c >= window or (n_seg == 0 and np.float32(c) >= first_min)):
                    if n_seg and run - last_y < seg_dist:
                        out[-1][1] = en
                    else:
                        out.append([run, en])
                        n_seg += 1
                    last_y = en
            run = max(run, last_open[lane])
        open_pos, state, last_word = run, cur, ins[31]
    return np.array(out, dtype=np.int64).reshape(-1, 2)


def _fixture_reads(npz):
    return [rd for _, rd in _fmt.load_npz(os.path.join(G, npz))]


# ---- tests --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_jnn", 0), ("synth_rna.npz", "ref_rna_jnn", 1),
                                              ("jnn_stalls_dna.npz", "ref_jnn_stalls_dna", 0),
                                              ("jnn_stalls_rna.npz", "ref_jnn_stalls_rna", 1)])
def test_reference_sets_equal_reference_stdout(ref, npz, txt, rna_flag):
    reads = _fmt.load_npz(os.path.join(G, npz))
    segs = [ref.jnn(rd[0], REFERENCE[rna_flag]) for _, rd in reads]
    for compact, suffix in ((False, ".txt"), (True, "_c.txt")):
        got = _fmt.JNN_HDR + "".join(_fmt.jnn_line(rid, len(rd[0]), segs[r], compact)
                                     for r, (rid, rd) in enumerate(reads))
        assert got == open(os.path.join(G, txt + suffix)).read(), suffix


@pytest.mark.parametrize("rna_flag", [0, 1])
def test_reference_sets_equal_orc_jnn(ref, rna_flag):
    orc = Oracle()
    win = REFERENCE[rna_flag][0]
    reads = stall_reads(np.random.default_rng(40 + rna_flag), 40, win) + \
        [(np.zeros(0, np.int16),), (np.array([700], np.int16),), (np.full(3000, 1300, np.int16),)]
    n_seg = 0
    for rd in reads:
        exp = orc.jnn(rd[0], rna_flag)
        assert np.array_equal(ref.jnn(rd[0], REFERENCE[rna_flag]), exp)
        n_seg += len(exp)
    assert n_seg > len(reads)


@pytest.mark.parametrize("seed", range(6))
def test_automaton_equals_counter_machine_for_random_sets(ref, seed):
    rng = np.random.default_rng(100 + seed)
    p = random_set(rng, automaton=True)
    if seed == 0:
        p = (p[0], p[1], 6, p[3], p[4], p[5])  # eight states: every 3-bit field of a map in use
    reads = _fixture_reads("jnn_stalls_dna.npz")[:6] + [rd[:1] for rd in stall_reads(rng, 6, p[0], scale=0.5)]
    n_seg = 0
    for rd in reads:
        exp = ref.jnn(rd[0], p)
        assert np.array_equal(walk(rd[0], p), exp), p
        assert ref.decrements(rd[0], p) == 0
        n_seg += len(exp)
    assert n_seg > 0, p


def test_smallest_window_fills_the_segment_slots(ref):
    """window 32, stall_len 1.0, error 0: stretches of 32 in-band samples closed by one outlier each -- n/33
    segments, against n/32 + 1 slots"""
    p = (32, 1.0, 0, 0, 1, 0.75)
    raw = np.tile(np.r_[np.full(32, 500, np.int16), np.int16(900)], 200)
    exp = ref.jnn(raw, p)
    assert len(exp) == len(raw) // 33
    assert len(exp) <= len(raw) // 32 + 1
    assert np.array_equal(walk(raw, p), exp)


def test_corrector_never_acts_when_error_below_corrector(ref):
    rng = np.random.default_rng(7)
    reads = _fixture_reads("jnn_stalls_dna.npz") + _fixture_reads("sp1_dna.npz")[:20] + \
        stall_reads(rng, 20, 200, outlier_every=1)
    sets = [CDNA_R9, DRNA_R9, (188, 0.25, 4, 60, 50, 0.7), (64, 0.5, 40, 50, 41, 0.75), (40, 1.0, 0, 0, 1, 1.2)]
    sets += [random_set(rng, automaton=True) for _ in range(4)]
    for p in sets:
        assert sum(ref.decrements(rd[0], p) for rd in reads) == 0, p


@pytest.mark.parametrize("p", [(64, 1.0, 2, 50, 0, 0.75), (150, 0.25, 50, 50, 50, 0.75), (188, 0.25, 40, 60, 10, 0.7)])
def test_corrector_acts_when_error_reaches_corrector(ref, p):
    """with error >= corrector the decrement fires and the segments differ from the rule "a stretch closes at its
    (error+1)-th outlier" (the same set with a corrector that cannot act)"""
    rng = np.random.default_rng(11)
    reads = stall_reads(rng, 30, p[0], outlier_every=1)
    no_corr = p[:4] + (INT32_MAX,) + p[5:]
    dec = differ = 0
    for rd in reads:
        d = ref.decrements(rd[0], p)
        dec += d
        if d:
            differ += int(not np.array_equal(ref.jnn(rd[0], p), ref.jnn(rd[0], no_corr)))
    assert dec > 0 and differ > 0, (dec, differ)
    if p[2] <= 6:
        for rd in reads[:5]:
            assert np.array_equal(walk(rd[0], no_corr), ref.jnn(rd[0], no_corr))

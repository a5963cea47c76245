"""GPU tests of SGPU_WANT_PREFIX with the caller's own sets (sgpu_set_prefix, Context.set_prefix): the reference's sets
given explicitly reproduce the default path and the reference's stdout; custom adaptor sets (windows of every residue
mod 8, 2 and 13,981, a 4 kHz window, odd windows, lo_thresh > hi_thresh, negative seg_dist and std_scale) and poly-A
sets on both routes (the automaton for error < corrector, the reference's counters for every other set) equal
orc_prefix_set (tests/tools/prefix_set_oracle.c) read by read; the other products of a batch do not change; a host slot
keeps the set in force at its submit; SGPU_PARAM_PORE is ignored while a set is in force; refused sets leave the
previous one in place. Positions and the float bits of all six statistics are compared exactly."""
import os

import numpy as np
import pytest

import _fmt
from _oracle import Oracle
from _prefix_ref import (ADAPTORS, AUTOMATON, EXACT, INT32_MAX, POLYA_R9, RNA_R9, PrefixSetRef, named_set,
                         random_set, set_read)
import sigtk_b200 as sg
from sigtk_b200 import _lib as _sl
from test_gpu_prefix import adaptor_read

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_INVAL = -1
ALL_WANTS = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
R9 = sg.Prefix(sg.Adaptor.RNA_R9, sg.Polya.R9)
RNA004 = sg.Prefix(sg.Adaptor.RNA004, sg.Polya.R9)


def as_prefix(p):
    return sg.Prefix(sg.Adaptor(*p[0]), sg.Polya(*p[1]))


@pytest.fixture(scope="module")
def ref():
    return PrefixSetRef()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 26, max_reads=12000) as c:
        yield c
        c.set_prefix(None)
        c.set_param(_sl.PARAM_PORE, 0)


@pytest.fixture(autouse=True)
def no_set_between_tests(ctx):
    ctx.set_prefix(None)
    ctx.set_param(_sl.PARAM_PORE, 0)
    yield
    ctx.set_prefix(None)
    ctx.set_param(_sl.PARAM_PORE, 0)


def bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def check(ref, pos, stat, reads, rna, p, what):
    """positions and statistics of every read against the restatement; -> (reads with an adaptor, with a poly-A)"""
    n_a = n_p = 0
    for r, rd in enumerate(reads):
        epos, est = ref.prefix(*rd, rna, p)
        got = np.asarray(pos[r], dtype=np.int64)
        assert np.array_equal(got, epos), f"{what}: read {r} of {len(rd[0])}: positions {got} != {epos}"
        assert np.array_equal(bits(stat[r]), bits(est)), f"{what}: read {r}: statistics {stat[r]} != {est}"
        n_a += epos[1] > 0
        n_p += epos[3] > 0
    return n_a, n_p


def same_prefix(a, b):
    return (np.array_equal(a.prefix_pos, b.prefix_pos) and
            np.array_equal(bits(a.prefix_stat), bits(b.prefix_stat)))


def same_other_products(a, b):
    """the outputs other than PREFIX of two host results of the same batch, by their bits"""
    for x, y in ((a.ev_off, b.ev_off), (a.ev_start, b.ev_start), (a.ev_mean, b.ev_mean), (a.ev_stdv, b.ev_stdv),
                 (a.stat, b.stat), (a.ent, b.ent)):
        if x is None or y is None or not np.array_equal(np.ascontiguousarray(x).view(np.uint8),
                                                        np.ascontiguousarray(y).view(np.uint8)):
            return False
    if len(a.jnn) != len(b.jnn) or not all(np.array_equal(p, q) for p, q in zip(a.jnn, b.jnn)):
        return False
    return all(np.array_equal(p.view(np.uint32), q.view(np.uint32)) for p, q in zip(a.pa, b.pa))


def device_prefix(torch, c, reads, rna):
    """sgpu_run_device on device copies of `reads`; -> (pos int32[n][4], stat float32[n][6])"""
    lens = np.array([len(rd[0]) for rd in reads], np.int64)
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    raw = np.zeros(max(int(off[-1]), 8), np.int16)
    for r, rd in enumerate(reads):
        raw[off[r]:off[r] + lens[r]] = rd[0]
    dev = torch.device("cuda:0")
    arrs = [torch.from_numpy(x).to(dev) for x in (
        raw, off, lens.astype(np.int32), np.array([np.float32(rd[2]) for rd in reads], np.float32),
        np.array([np.float32(rd[3]) / np.float32(rd[1]) for rd in reads], np.float32))]
    torch.cuda.synchronize()
    d = c.run_device(*[a.data_ptr() for a in arrs], len(reads), int(off[-1]), rna, sg.WANT_PREFIX,
                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert c.counters()["status"] == 0
    n = len(reads)
    return c.d2h(d.prefix_pos, np.int32, 4 * n).reshape(n, 4), c.d2h(d.prefix_stat, np.float32, 6 * n).reshape(n, 6)


def around_window(p, seed):
    """reads of window - 1 .. window + 2 samples (cut from a read with an adaptor at its start)"""
    aw = p[0][0]
    base = set_read(0, seed, p)
    return [(base[0][:n].copy(),) + base[1:] for n in range(max(aw - 1, 0), aw + 3)]


# ---- the reference's sets given explicitly ---------------------------------------------------------------------------
@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_prefix_stat.txt", 0),
                                              ("synth_rna.npz", "ref_rna_prefix_stat.txt", 1),
                                              ("prefix_adaptor_dna.npz", "ref_prefix_adaptor_dna_stat.txt", 0),
                                              ("prefix_adaptor_rna.npz", "ref_prefix_adaptor_rna_stat.txt", 1)])
def test_explicit_r9_set_is_the_default(ctx, orc, npz, txt, rna_flag):
    """int16, svb-zd and device-resident batches; the set in force makes SGPU_PARAM_PORE = 1 ineffective"""
    torch = pytest.importorskip("torch")
    named = _fmt.load_npz(os.path.join(G, npz))
    reads = [rd for _, rd in named]
    svb = [(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads]
    default = ctx.run(reads, rna=rna_flag, want=sg.WANT_PREFIX)
    ctx.set_prefix(R9)
    ctx.set_param(_sl.PARAM_PORE, 1)
    got = ctx.run(reads, rna=rna_flag, want=sg.WANT_PREFIX)
    assert same_prefix(got, default)
    assert same_prefix(ctx.run_svbzd(svb, rna=rna_flag, want=sg.WANT_PREFIX), default)
    dpos, dst = device_prefix(torch, ctx, reads, rna_flag)
    assert np.array_equal(dpos, default.prefix_pos) and np.array_equal(bits(dst), bits(default.prefix_stat))
    rows = [(rid, len(rd[0]), got.prefix_pos[r], got.prefix_stat[r]) for r, (rid, rd) in enumerate(named)]
    text = _fmt.PREFIX_HDR + _fmt.PREFIX_HDR_STAT + "\n" + "".join(_fmt.prefix_line(r, n, p, s, True) for r, n, p, s in rows)
    assert text == open(os.path.join(G, txt)).read()
    if rna_flag == 0 and npz == "sp1_dna.npz":
        text = _fmt.PREFIX_HDR + "\n" + "".join(_fmt.prefix_line(r, n, p, s) for r, n, p, s in rows)
        assert text == open(os.path.join(G, "prefix_dna.exp")).read()


@pytest.mark.parametrize("rna_flag", [0, 1])
def test_explicit_rna004_set_is_the_default(ctx, orc, ref, rna_flag):
    """RNA004's set given explicitly equals SGPU_PARAM_PORE = 1 without a set (int16, svb-zd, device-resident) and
    orc_adaptor_polya_pore; under PORE = 0 too"""
    torch = pytest.importorskip("torch")
    reads = [adaptor_read(k, int(n), seed=17) for k, n in enumerate([30000, 45000, 60000, 90000, 25000, 150000, 33333])]
    reads += [set_read(k, 19, (sg.Adaptor.RNA004, sg.Polya.R9)) for k in range(20)]
    svb = [(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads]
    ctx.set_param(_sl.PARAM_PORE, 1)
    default = ctx.run(reads, rna=rna_flag, want=sg.WANT_PREFIX)
    for r, rd in enumerate(reads):
        pos, st = orc.adaptor_polya(*rd, rna=rna_flag, pore=1)
        assert np.array_equal(default.prefix_pos[r].astype(np.int64), pos)
        assert np.array_equal(bits(default.prefix_stat[r]), bits(st))
    ctx.set_param(_sl.PARAM_PORE, 0)
    ctx.set_prefix(RNA004)
    assert same_prefix(ctx.run(reads, rna=rna_flag, want=sg.WANT_PREFIX), default)
    assert same_prefix(ctx.run_svbzd(svb, rna=rna_flag, want=sg.WANT_PREFIX), default)
    dpos, dst = device_prefix(torch, ctx, reads, rna_flag)
    assert np.array_equal(dpos, default.prefix_pos) and np.array_equal(bits(dst), bits(default.prefix_stat))
    assert check(ref, default.prefix_pos, default.prefix_stat, reads, rna_flag, tuple(RNA004), "rna004")[0] >= 20


# ---- custom sets -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(ADAPTORS) + sorted(AUTOMATON) + sorted(EXACT))
def test_custom_set_vs_restatement(ctx, ref, name):
    """seeded reads with stretches scaled to the set, reads of window - 1 .. window + 2 samples, reads without a
    poly-A; every other product of an all-wants batch bit for bit as without the set"""
    p = named_set(name)
    seed = 100 + (sorted(ADAPTORS) + sorted(AUTOMATON) + sorted(EXACT)).index(name)
    reads = [set_read(k, seed, p) for k in range(48)] + [set_read(k, seed + 1, p, polya=False) for k in range(4)]
    reads += around_window(p, seed + 2)
    base = ctx.run(reads, rna=1, want=ALL_WANTS)
    ctx.set_prefix(as_prefix(p))
    res = ctx.run(reads, rna=1, want=ALL_WANTS)
    n_a, n_p = check(ref, res.prefix_pos, res.prefix_stat, reads, 1, p, name)
    assert same_other_products(res, base)
    if name not in ("lo_above_hi", "smallest"):   # (a window of 2 samples follows the noise too)
        assert n_a >= len(reads) // 2, n_a
    if name not in ("lo_above_hi", "error_max", "smallest"):
        assert n_p >= len(reads) // 2, n_p
    # without rna: the adaptor only
    res0 = ctx.run(reads[:16], rna=0, want=sg.WANT_PREFIX)
    check(ref, res0.prefix_pos, res0.prefix_stat, reads[:16], 0, p, name + " dna")


@pytest.mark.parametrize("aw", list(range(2000, 2008)) + [9, 15, 333])
def test_adaptor_window_residues(ctx, ref, aw):
    """windows of every residue mod 8 (the upper range of a window difference at every alignment) and short odd ones"""
    p = ((aw, 0.5, max(aw * 3 // 4, 1), max(aw, 100), 200000), POLYA_R9)
    reads = [set_read(k, 300 + aw, p) for k in range(24)] + around_window(p, 400 + aw)
    ctx.set_prefix(as_prefix(p))
    res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    n_a, n_p = check(ref, res.prefix_pos, res.prefix_stat, reads, 1, p, f"window {aw}")
    assert n_a >= 12 and n_p >= 12, (n_a, n_p)


@pytest.mark.parametrize("name", ["w4k", "error32", "corrector0"])
def test_long_read_svbzd_and_device(ctx, orc, ref, name):
    """a read of 2,000,000 samples among set-scaled ones, as int16 records, svb-zd streams and device-resident"""
    torch = pytest.importorskip("torch")
    p = named_set(name)
    reads = [set_read(0, 500, p, n=2_000_000)] + [set_read(k, 501, p) for k in range(1, 12)]
    ctx.set_prefix(as_prefix(p))
    res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    n_a, _ = check(ref, res.prefix_pos, res.prefix_stat, reads, 1, p, name)
    assert n_a >= 6
    assert same_prefix(ctx.run_svbzd([(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads], rna=1,
                                     want=sg.WANT_PREFIX), res)
    dpos, dst = device_prefix(torch, ctx, reads, 1)
    assert np.array_equal(dpos, res.prefix_pos) and np.array_equal(bits(dst), bits(res.prefix_stat))


@pytest.mark.parametrize("exact", [False, True])
def test_more_reads_than_warps(ctx, ref, exact):
    """10,000 reads: more than prefix_walk's 148 * 16 blocks of four warps, so that warps take several reads"""
    rng = np.random.default_rng(61 + exact)
    p = (300, 0.5, 200, 100, 50000), random_set(rng, exact)[1]
    p = (p[0], (60, p[1][1], p[1][2], p[1][3], p[1][4]))
    reads = [set_read(k, 62 + exact, p, n=int(rng.integers(1500, 3500))) for k in range(10000)]
    ctx.set_prefix(as_prefix(p))
    res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    n_a, n_p = check(ref, res.prefix_pos, res.prefix_stat, reads, 1, p, "many reads")
    assert n_a > 5000, n_a


# ---- when the set takes effect ---------------------------------------------------------------------------------------
def test_slot_keeps_the_set_of_its_submit(ctx, ref, orc):
    a, b = named_set("w4k"), named_set("corrector0")
    reads = [set_read(k, 81, a) for k in range(20)] + [set_read(k, 82, b) for k in range(20)]
    ctx.set_prefix(as_prefix(a))
    ctx.fill(0, reads, 1)
    ctx.submit(0, sg.WANT_PREFIX)
    ctx.set_prefix(as_prefix(b))
    ctx.fill(1, reads, 1)
    ctx.submit(1, sg.WANT_PREFIX)
    ctx.set_prefix(None)
    r0, r1 = ctx.wait(0, sg.WANT_PREFIX), ctx.wait(1, sg.WANT_PREFIX)
    check(ref, r0.prefix_pos, r0.prefix_stat, reads, 1, a, "slot 0")
    check(ref, r1.prefix_pos, r1.prefix_stat, reads, 1, b, "slot 1")
    assert not np.array_equal(r0.prefix_pos, r1.prefix_pos)
    # PORE is ignored while a set is in force and applies again after set_prefix(None)
    ctx.set_prefix(R9)
    ctx.set_param(_sl.PARAM_PORE, 1)
    with_set = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    check(ref, with_set.prefix_pos, with_set.prefix_stat, reads, 1, tuple(R9), "R9 set under PORE 1")
    ctx.set_prefix(None)
    res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    for r, rd in enumerate(reads):
        pos, st = orc.adaptor_polya(*rd, rna=1, pore=1)
        assert np.array_equal(res.prefix_pos[r].astype(np.int64), pos), f"after set_prefix(None): read {r}"
        assert np.array_equal(bits(res.prefix_stat[r]), bits(st))


# ---- refusals and boundaries -------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [
    ((1, 0.5, 1500, 2000, 200000), POLYA_R9),               # adaptor window < 2
    ((0, 0.5, 1500, 2000, 200000), POLYA_R9),
    ((-2000, 0.5, 1500, 2000, 200000), POLYA_R9),
    ((13982, 0.5, 1500, 2000, 200000), POLYA_R9),           # 1200 * window > 2^24
    ((INT32_MAX, 0.5, 1500, 2000, 200000), POLYA_R9),
    ((2000, float("nan"), 1500, 2000, 200000), POLYA_R9),   # std_scale not finite
    ((2000, float("inf"), 1500, 2000, 200000), POLYA_R9),
    ((2000, float("-inf"), 1500, 2000, 200000), POLYA_R9),
    (RNA_R9, (250, 1.0, -1, 200, 50)),                      # error < 0
    (RNA_R9, (250, 1.0, 30, 200, -1)),                      # corrector < 0
    (RNA_R9, (250, float("nan"), 30, 200, 50)),             # stall_len not finite
    (RNA_R9, (250, float("-inf"), 30, 200, 50)),
])
def test_refused_set_keeps_the_previous(ctx, ref, bad):
    keep = named_set("error_above")
    ctx.set_prefix(as_prefix(keep))
    with pytest.raises(sg.SgpuError) as e:
        ctx.set_prefix(as_prefix(bad))
    assert e.value.code == E_INVAL
    reads = [set_read(k, 91, keep) for k in range(12)]
    res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
    check(ref, res.prefix_pos, res.prefix_stat, reads, 1, keep, "after a refusal")


def test_boundary_sets_are_accepted(ctx, ref):
    sets = [((2, 0.5, 1500, 600, 200000), POLYA_R9), ((13981, 0.5, 9000, 4000, 900000), POLYA_R9),
            ((2000, 0.0, -(2**31), 1, INT32_MAX), (250, 1.0, 0, 200, 0)),
            (RNA_R9, (-(2**31), 0.0, INT32_MAX, -(2**31), INT32_MAX)),
            (RNA_R9, (INT32_MAX, -3.0, 0, INT32_MAX, 1)),
            ((2000, -1e30, 1500, 2000, 200000), (250, 1e30, 5, 200, 6))]
    for p in sets:
        reads = [set_read(k, 95, p) for k in range(8)]
        ctx.set_prefix(as_prefix(p))
        res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
        check(ref, res.prefix_pos, res.prefix_stat, reads, 1, p, f"boundary {p}")

"""GPU tests of the ordered float sums and of the median select at their edges (float_order.cuh, stat.cu, prefix.cu):
`sigtk stat` (all six numbers), the jnn band (through the jnn segments) and the prefix statistics on the crafted corpus
of tests/_stat_corpus.py, against the plain reference of tests/_stat_ref.py and the oracle, bit for bit, with both
roles of the moments kernel (PARAM_STAT_CTA_MIN 0: one CTA per read; the default; 2^31: one warp per read). Padding
after a read must not matter: garbage past read_len in a device-resident batch, stale samples of an earlier batch in
a host slot."""
import numpy as np
import pytest

from _device_out import assert_same, collect
import _stat_corpus as K
import _stat_ref as R
from _oracle import Oracle
from _prefix_ref import PrefixSetRef
import sigtk_b200 as sg
from sigtk_b200 import _lib as _sl

pytestmark = pytest.mark.gpu
ALL_WANTS = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
CTA_MIN_DEFAULT = 131072
CORPUS = K.corpus()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ref():
    return PrefixSetRef()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 23, max_reads=4096) as c:
        yield c


@pytest.fixture(autouse=True)
def defaults(ctx):
    yield
    ctx.set_param(_sl.PARAM_STAT_CTA_MIN, CTA_MIN_DEFAULT)
    ctx.set_prefix(None)


@pytest.fixture(scope="module")
def corpus_want(orc):
    """per read: the plain reference's six numbers, the oracle's, the oracle's jnn segments"""
    return [(R.stat(*rd), orc.stat(*rd), orc.jnn(rd[0], 0)) for _, rd, _ in CORPUS]


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("cta_min", [0, CTA_MIN_DEFAULT, 1 << 31])
def test_corpus_stat_and_jnn(ctx, corpus_want, cta_min):
    for _, _, check in CORPUS:
        check()
    ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
    res = ctx.run([rd for _, rd, _ in CORPUS], rna=0, want=sg.WANT_STAT | sg.WANT_JNN)
    bad = []
    for r, ((name, rd, _), (plain, oracle, jnn)) in enumerate(zip(CORPUS, corpus_want)):
        if not (R.same_stat(res.stat[r], plain) and R.same_stat(res.stat[r], oracle)):
            bad.append(f"{name}: stat {res.stat[r]} != {plain}")
        if not np.array_equal(res.jnn[r], jnn):
            bad.append(f"{name}: jnn {res.jnn[r][:4]} != {jnn[:4]}")
    assert not bad, bad


def median_batch():
    return K.median_reads() + K.degenerate_units()


@pytest.mark.parametrize("cta_min", [0, CTA_MIN_DEFAULT])
def test_median_edges(ctx, orc, cta_min):
    """medians by the 1,024-thread select (cta_min 0) and by the 256-thread one; a zero pA median is pA(raw median)
    (its sign is not pinned by the reference, DESIGN section 4: the oracle's only has to be a zero too)"""
    reads = median_batch()
    ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
    res = ctx.run([rd for _, rd in reads], rna=0, want=sg.WANT_STAT)
    for r, (name, rd) in enumerate(reads):
        got, plain = res.stat[r], R.stat(*rd)
        if K.mixed_zero(name):
            assert R.same_stat(got[:5], plain[:5]) and got[5] == 0 and orc.stat(*rd)[5] == 0, name
            assert bits(got[5]) == bits(R.pa(np.array([got[4]], np.int16), *rd[1:])[0]), name
        else:
            assert R.same_stat(got, plain) and R.same_stat(got, orc.stat(*rd)), f"{name}: {got} != {plain}"


@pytest.mark.parametrize("sign", [1.0, -1.0])
@pytest.mark.parametrize("rna", [0, 1])
def test_prefix_stretches_at_every_residue(ctx, ref, sign, rna):
    """the adaptor's and the poly-A's mean, stdv and median (the unaligned select on sub-ranges, rank from the other
    end for a negative unit) against orc_prefix_set and the plain reference"""
    reads = K.prefix_reads(sign)
    ctx.set_prefix(sg.Prefix(sg.Adaptor(*K.PREFIX_SET[0]), sg.Polya(*K.PREFIX_SET[1])))
    res = ctx.run(reads, rna=rna, want=sg.WANT_PREFIX)
    for r, rd in enumerate(reads):
        pos, st = ref.prefix(*rd, rna, K.PREFIX_SET)
        assert pos[1] > 0 and (pos[3] > 0 or not rna or sign < 0)
        assert np.array_equal(res.prefix_pos[r].astype(np.int64), pos), f"read {r}: {res.prefix_pos[r]} != {pos}"
        assert np.array_equal(bits(res.prefix_stat[r]), bits(st)), f"read {r}: {res.prefix_stat[r]} != {st}"
        p = R.pa(*rd)[pos[0]:pos[1]]
        assert R.same_stat(res.prefix_stat[r][:3], [R.meanf(p), R.stdvf(p), R.rank_half(p)])


# ---- padding -----------------------------------------------------------------------------------------------------------
def padding_reads():
    """lengths of every residue mod 8: the n = 1 .. 17 median reads, crafted sums, prefix reads"""
    reads = [rd for _, rd in K.median_reads() if len(rd[0]) < 300]
    reads += [rd for name, rd, _ in CORPUS if name.startswith(("band_edges", "hit_", "cross_", "len_8191", "len_33"))]
    reads += K.prefix_reads(1.0)[:8] + K.prefix_reads(-1.0)[:4]
    assert {len(rd[0]) % 8 for rd in reads} == set(range(8))
    return reads


def garbage(k, rd, m):
    """m samples past a read: full-scale values, LOW ones (pA <= 0 for the read's offset), the read's median bin"""
    med = int(np.sort(rd[0])[len(rd[0]) // 2])
    low = int(np.clip(-np.float32(rd[2]) - 7, -32768, 32767))
    pat = [(32767, -32768), (low, low), (med, med - 1), (med + 1, 0), (-32768, med)][k % 5]
    return np.resize(np.clip(np.array(pat, np.int64), -32768, 32767).astype(np.int16), m)


def device_run(torch, c, reads, pad, rna, want):
    lens = np.array([len(rd[0]) for rd in reads], np.int64)
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(int(off[-1]), np.int16)
    for r, rd in enumerate(reads):
        flat[off[r]:off[r] + lens[r]] = rd[0]
        if pad:
            flat[off[r] + lens[r]:off[r + 1]] = garbage(r, rd, int(off[r + 1] - off[r] - lens[r]))
    dev = torch.device("cuda:0")
    arrs = [torch.from_numpy(x).to(dev) for x in (
        flat, off, lens.astype(np.int32), np.array([np.float32(rd[2]) for rd in reads], np.float32),
        np.array([np.float32(rd[3]) / np.float32(rd[1]) for rd in reads], np.float32))]
    torch.cuda.synchronize()
    d = c.run_device(*[a.data_ptr() for a in arrs], len(reads), int(off[-1]), rna, want,
                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert c.counters()["status"] == 0
    return collect(c, d, len(reads), off, lens, want, int(off[-1]))


@pytest.mark.parametrize("rna", [0, 1])
def test_device_padding_does_not_matter(ctx, rna):
    torch = pytest.importorskip("torch")
    reads = padding_reads()
    ctx.set_prefix(sg.Prefix(sg.Adaptor(*K.PREFIX_SET[0]), sg.Polya(*K.PREFIX_SET[1])))
    clean = device_run(torch, ctx, reads, False, rna, ALL_WANTS)
    dirty = device_run(torch, ctx, reads, True, rna, ALL_WANTS)
    assert_same(dirty, clean, "garbage padding")
    st = clean["stat"].view(np.float32).reshape(-1, 6)
    for r, rd in enumerate(reads):
        assert R.same_stat(st[r], R.stat(*rd)), f"read {r} (n={len(rd[0])})"


def test_device_pa_padding_does_not_matter(ctx):
    torch = pytest.importorskip("torch")
    reads = padding_reads()
    sigs = [R.pa(*rd) for rd in reads]
    lens = np.array([len(s) for s in sigs], np.int64)
    off = np.zeros(len(sigs) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    junk = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38, 0.0, 1e-40], np.float32)
    outs = []
    for pad in (False, True):
        flat = np.zeros(int(off[-1]), np.float32)
        for r, s in enumerate(sigs):
            flat[off[r]:off[r] + lens[r]] = s
            if pad:
                flat[off[r] + lens[r]:off[r + 1]] = np.resize(np.roll(junk, r), int(off[r + 1] - off[r] - lens[r]))
        dev = torch.device("cuda:0")
        a = [torch.from_numpy(x).to(dev) for x in (flat, off, lens.astype(np.int32))]
        torch.cuda.synchronize()
        d = ctx.run_device_pa(a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), len(sigs), int(off[-1]), 0,
                              sg.WANT_EVENTS, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert ctx.counters()["status"] == 0
        outs.append(collect(ctx, d, len(sigs), off, lens, sg.WANT_EVENTS, int(off[-1])))
    assert_same(outs[1], outs[0], "garbage pA padding")


def test_host_slot_stale_padding(ctx):
    """a batch of extreme reads, then in the same slot a batch whose padding still holds their samples: the results
    equal those of a fresh context"""
    reads = padding_reads()
    span = sum((len(rd[0]) + 7) // 8 * 8 for rd in reads)
    ext = np.resize(np.array([32767, -32768, 16, 15, 592, 591, 1023, 1024], np.int16), span + 64)
    ctx.set_prefix(sg.Prefix(sg.Adaptor(*K.PREFIX_SET[0]), sg.Polya(*K.PREFIX_SET[1])))
    ctx.run([(ext, 8192.0, 3.0, 1402.882324)], rna=1, want=ALL_WANTS)
    got = ctx.run(reads, rna=1, want=ALL_WANTS)
    with sg.Context(device=0, max_samples=1 << 23, max_reads=4096) as fresh:
        fresh.set_prefix(sg.Prefix(sg.Adaptor(*K.PREFIX_SET[0]), sg.Polya(*K.PREFIX_SET[1])))
        want = fresh.run(reads, rna=1, want=ALL_WANTS)
    for k in ("ev_off", "ev_start", "stat", "ent", "prefix_pos", "prefix_stat"):
        assert np.array_equal(np.ascontiguousarray(getattr(got, k)).view(np.uint8),
                              np.ascontiguousarray(getattr(want, k)).view(np.uint8)), k
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(got.pa, want.pa))
    assert all(np.array_equal(a, b) for a, b in zip(got.jnn, want.jnn))
    for r, rd in enumerate(reads):
        assert R.same_stat(got.stat[r], R.stat(*rd)), f"read {r} (n={len(rd[0])})"

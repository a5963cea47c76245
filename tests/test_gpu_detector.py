"""Event detection with the caller's own detector parameters (sgpu_set_detector), on the GPU.

A reference set given explicitly runs on the general route (the route of pA records) and must give the default path's
events bit for bit, for int16 slots, svb-zd streams, device-resident runs, pA records and live entries of both forms.
Any other set must give the oracle's composition (tests/_detector_sets.py, test_detector_sets.py) bit for bit, on short,
empty and 2,000,000-sample reads, in batches that run every grid-stride loop more than once, and on pA with NaN and
Inf. Live reads keep the set of their START entry."""
import numpy as np
import pytest

from _detector_ref import stream_reference, whole_read
from _detector_sets import CUSTOM, REFERENCE
from _live_ref import concat, same_events, split_lengths
from _oracle import Oracle
from test_gpu_live import device_push, tables
from test_gpu_live_pa import device_push_pa
from test_gpu_pa_input import run_device as run_device_pa
from test_live_contract import golden
import sigtk_b200 as sg
from sigtk_b200 import synth

gpu = pytest.mark.gpu

E_INVAL = -1
START, END, RNA = sg.LIVE_START, sg.LIVE_END, sg.LIVE_RNA
ALL_SETS = {"dna": REFERENCE[0], "rna": REFERENCE[1], **CUSTOM}


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 23, max_reads=4096) as c:
        c.live_open(256)
        yield c
        c.set_detector(None)


@pytest.fixture(autouse=True)
def no_set_between_tests(ctx):
    ctx.set_detector(None)
    yield
    ctx.set_detector(None)


def same(a, b):
    """two (start, length, mean, stdv) tuples: the same boundaries, NaN in the same places, every other float by its
    bits"""
    if not np.array_equal(np.asarray(a[0], np.uint64), np.asarray(b[0], np.uint64)):
        return False
    for j in (1, 2, 3):
        x, y = np.asarray(a[j], np.float32), np.asarray(b[j], np.float32)
        if x.shape != y.shape or not np.array_equal(np.isnan(x), np.isnan(y)):
            return False
        if not np.array_equal(x[~np.isnan(x)].view(np.uint32), y[~np.isnan(y)].view(np.uint32)):
            return False
    return True


def ev(res, r):
    t = res.events(r)
    return t.start, t.length, t.mean, t.stdv


def check_truth(orc, res, signals, params, what):
    for r, pa in enumerate(signals):
        assert same(ev(res, r), whole_read(orc, pa, 0, params=params)), f"{what}: read {r} of {len(pa)} samples"


def same_tables(a, b):
    return (np.array_equal(a.ev_off, b.ev_off) and np.array_equal(a.ev_start, b.ev_start) and
            np.array_equal(a.ev_mean.view(np.uint32), b.ev_mean.view(np.uint32)) and
            np.array_equal(a.ev_stdv.view(np.uint32), b.ev_stdv.view(np.uint32)))


def mixed_reads(seed):
    """short reads (below 2 w for every set), an empty read, synthetic and real reads"""
    rng = np.random.default_rng(seed)
    out = [synth.make_read_cb(k, n, seed=seed) for k, n in enumerate((0, 1, 2, 3, 5, 13, 27, 28, 29, 600, 7000))]
    out += synth.make_reads(6, mean=30000.0, seed=seed)
    out += golden("sp1_dna.npz")[int(rng.integers(0, 80)):][:10]
    return out


def device_run(torch, c, reads, rna, want=sg.WANT_EVENTS):
    """sgpu_run_device on device copies of int16 `reads`; -> a BatchResult with the event outputs"""
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
    d = c.run_device(*[a.data_ptr() for a in arrs], len(reads), int(off[-1]), rna, want,
                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    cnt = c.counters()
    assert cnt["status"] == 0
    n, ne = len(reads), cnt["n_events"]
    res = sg.BatchResult(n_reads=n, read_len=lens.astype(np.uint32))
    res.ev_off = c.d2h(d.ev_off, np.uint64, n + 1)
    res.ev_start = c.d2h(d.ev_start, np.uint32, ne)
    res.ev_mean = c.d2h(d.ev_mean, np.float32, ne)
    res.ev_stdv = c.d2h(d.ev_stdv, np.float32, ne)
    res.fixups = c.d2h(d.fixups, np.uint32, n)
    return res


# ---- the reference's sets given explicitly ---------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("rna", [0, 1])
def test_explicit_reference_set_is_the_default_path(ctx, orc, rna):
    torch = pytest.importorskip("torch")
    reads = (golden("sp1_dna.npz") if rna == 0 else golden("synth_rna.npz")) + synth.make_reads(40, seed=9 + rna, rna=bool(rna))
    pa = [orc.pa(*rd) for rd in reads]
    svb = [(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads]
    runs = {}
    for name, det in (("default", None), ("explicit", sg.Detector(*REFERENCE[rna]))):
        ctx.set_detector(det)
        runs[name] = (ctx.run(reads, rna=rna), ctx.run_svbzd(svb, rna=rna), ctx.run_pa(pa, rna=rna),
                      device_run(torch, ctx, reads, rna), run_device_pa(torch, ctx, pa, rna))
    for k, what in enumerate(("int16", "svb-zd", "pA", "device int16", "device pA")):
        assert same_tables(runs["default"][k], runs["explicit"][k]), what
    assert int(runs["explicit"][0].ev_off[-1]) > 1000


# ---- other sets against the oracle -----------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", sorted(CUSTOM))
def test_custom_sets_on_every_input(ctx, orc, name):
    torch = pytest.importorskip("torch")
    params = CUSTOM[name]
    reads = mixed_reads(sorted(CUSTOM).index(name))
    pa = [orc.pa(*rd) for rd in reads]
    ctx.set_detector(sg.Detector(*params))
    for rna in (0, 1):  # rna no longer chooses the event parameters
        check_truth(orc, ctx.run(reads, rna=rna), pa, params, f"{name} int16 rna={rna}")
    check_truth(orc, ctx.run_svbzd([(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads], rna=0), pa,
                params, f"{name} svb-zd")
    check_truth(orc, device_run(torch, ctx, reads, 1), pa, params, f"{name} device int16")
    rng = np.random.default_rng(5)
    floats = pa + [(rng.normal(0, 1, 4000) * 1e-3).astype(np.float32), np.full(3000, 87.5, np.float32)]
    check_truth(orc, ctx.run_pa(floats, rna=0), floats, params, f"{name} pA")
    check_truth(orc, run_device_pa(torch, ctx, floats, 1), floats, params, f"{name} device pA")
    if name == "silent":
        res = ctx.run(reads, rna=0)
        assert all(res.events(r).n == (1 if len(rd[0]) else 0) for r, rd in enumerate(reads))


@gpu
@pytest.mark.parametrize("name", ["long_below_short", "dense"])
def test_huge_reads_and_batches_past_the_grids(orc, name):
    """two 2,000,000-sample reads, and 6,000 reads: more than the warps and CTAs of every kernel of the route"""
    params = CUSTOM[name]
    rng = np.random.default_rng(21)
    huge = [synth.make_read(k, 2_000_000, seed=4) for k in range(2)]
    many = [synth.make_read_cb(k, int(n), seed=6) for k, n in enumerate(rng.integers(0, 2000, 6000))]
    with sg.Context(device=0, max_samples=1 << 24, max_reads=8192) as c:
        c.set_detector(sg.Detector(*params))
        for reads in (huge, many):
            res = c.run(reads, rna=0)
            check_truth(orc, res, [orc.pa(*rd) for rd in reads], params, name)


@gpu
def test_nan_and_inf_in_pa(ctx, orc):
    rng = np.random.default_rng(8)
    signals = []
    for k in range(12):
        x = (rng.normal(80, 5, 3000)).astype(np.float32)
        x[rng.integers(0, 3000, 3)] = [np.nan, np.inf, -np.inf][k % 3]
        signals.append(x)
    signals.append(np.full(500, np.nan, np.float32))
    for params in (REFERENCE[0], CUSTOM["long_below_short"], CUSTOM["negative_height"], CUSTOM["windows_14_2"]):
        ctx.set_detector(sg.Detector(*params))
        check_truth(orc, ctx.run_pa(signals, rna=0), signals, params, f"NaN / Inf {params}")
    ctx.set_detector(None)
    default = ctx.run_pa(signals, rna=0)
    ctx.set_detector(sg.Detector(*REFERENCE[0]))
    explicit = ctx.run_pa(signals, rna=0)
    for r in range(len(signals)):
        assert same(ev(default, r), ev(explicit, r)), r


# ---- the setting's rules -----------------------------------------------------------------------------------------------
@gpu
def test_other_products_do_not_change(ctx):
    reads = synth.make_reads(10, seed=3)
    want = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
    a = ctx.run(reads, rna=1, want=want)
    ctx.set_detector(sg.Detector(*CUSTOM["dense"]))
    b = ctx.run(reads, rna=1, want=want)
    assert not same_tables(a, b)
    for k in ("stat", "ent", "prefix_pos", "prefix_stat"):
        assert np.array_equal(getattr(a, k).view(np.uint8), getattr(b, k).view(np.uint8)), k
    for r in range(len(reads)):
        assert np.array_equal(a.jnn[r], b.jnn[r]) and np.array_equal(a.pa[r].view(np.uint32), b.pa[r].view(np.uint32))


@gpu
def test_validation_and_null(ctx, orc):
    reads = synth.make_reads(4, seed=12)
    pa = [orc.pa(*rd) for rd in reads]
    good = CUSTOM["long_below_short"]
    ctx.set_detector(sg.Detector(*good))
    bad = [(1, 6, 1.4, 9.0, 0.2), (3, 1, 1.4, 9.0, 0.2), (15, 6, 1.4, 9.0, 0.2), (3, 15, 1.4, 9.0, 0.2),
           (0, 0, 1.4, 9.0, 0.2), (3, 6, np.nan, 9.0, 0.2), (3, 6, 1.4, np.inf, 0.2), (3, 6, 1.4, 9.0, -np.inf),
           (3, 6, 1.4, 9.0, np.nan)]
    for p in bad:
        with pytest.raises(sg.SgpuError) as e:
            ctx.set_detector(sg.Detector(*p))
        assert e.value.code == E_INVAL, p
    check_truth(orc, ctx.run(reads, rna=0), pa, good, "the set before the refused calls")
    ctx.set_detector(sg.Detector(2, 14, 1.0, 1.0, 0.0))  # the ends of the window range
    check_truth(orc, ctx.run(reads, rna=0), pa, (2, 14, 1.0, 1.0, 0.0), "windows 2 and 14")
    ctx.set_detector(None)
    check_truth(orc, ctx.run(reads, rna=1), pa, REFERENCE[1], "NULL: the reference's set for rna")


@gpu
def test_two_slots_in_flight_keep_their_sets(ctx, orc):
    reads = synth.make_reads(8, seed=13)
    pa = [orc.pa(*rd) for rd in reads]
    a, b = CUSTOM["long_below_short"], CUSTOM["short_wider"]
    ctx.set_detector(sg.Detector(*a))
    ctx.fill(0, reads, 0)
    ctx.submit(0, sg.WANT_EVENTS)
    ctx.set_detector(sg.Detector(*b))
    ctx.fill(1, reads, 0)
    ctx.submit(1, sg.WANT_EVENTS)
    ctx.set_detector(None)
    check_truth(orc, ctx.wait(0, sg.WANT_EVENTS), pa, a, "slot 0")
    check_truth(orc, ctx.wait(1, sg.WANT_EVENTS), pa, b, "slot 1")


# ---- live entries ----------------------------------------------------------------------------------------------------
def live_stream(ctx, signals, reads, form, rng, flags_rna=0):
    """every read on its own channel in seeded random splits; -> the tables each read's entries report, the splits"""
    splits = [split_lengths(len(s), rng) for s in signals]
    out = [[None] * len(s) for s in splits]
    at = [0] * len(signals)
    for k in range(max(len(s) for s in splits)):
        push, who = [], []
        for r, s in enumerate(splits):
            if k >= len(s):
                continue
            f = (START | flags_rna if k == 0 else 0) | (END if k == len(s) - 1 else 0)
            m = s[k]
            if form == "pa":
                push.append((r, f, signals[r][at[r]:at[r] + m]))
            else:
                rd = reads[r]
                push.append((r, f, rd[0][at[r]:at[r] + m], rd[1], rd[2], rd[3]))
            who.append(r)
            at[r] += m
        got = tables(ctx.live_push_pa(push) if form == "pa" else ctx.live_push(push))
        for r, t in zip(who, got):
            out[r][k] = t
    return out, splits


def live_reads(orc):
    reads = [synth.make_read_cb(k, n, seed=2) for k, n in enumerate((0, 1, 5, 13, 27, 28, 29, 600, 7000, 20000))]
    reads += golden("sp1_dna.npz")[:20]
    return reads, [orc.pa(*rd) for rd in reads]


@gpu
@pytest.mark.parametrize("form", ["int16", "pa"])
@pytest.mark.parametrize("name", sorted(ALL_SETS))
def test_live_entries_with_a_set(ctx, orc, form, name):
    params = ALL_SETS[name]
    reads, signals = live_reads(orc)
    rng = np.random.default_rng(sorted(ALL_SETS).index(name) + (100 if form == "pa" else 0))
    ctx.set_detector(sg.Detector(*params))
    got, splits = live_stream(ctx, signals, reads, form, rng, flags_rna=RNA)  # (RNA no longer chooses)
    for r, pa in enumerate(signals):
        ref, _ = stream_reference(orc, pa, 0, splits[r], params=params)
        for k in range(len(splits[r])):
            assert same_events(got[r][k], ref[k]), f"{name} {form}: read {r} chunk {k} of {splits[r][:6]}"
    if name in ("dna", "rna"):  # the same splits without a set: the default live path
        ctx.set_detector(None)
        rng = np.random.default_rng(sorted(ALL_SETS).index(name) + (100 if form == "pa" else 0))
        default, splits2 = live_stream(ctx, signals, reads, form, rng, flags_rna=RNA if name == "rna" else 0)
        assert splits2 == splits
        for r in range(len(signals)):
            for k in range(len(splits[r])):
                assert same_events(default[r][k], got[r][k]), f"{name} {form}: read {r} chunk {k}"


@gpu
@pytest.mark.parametrize("form", ["int16", "pa"])
def test_live_read_keeps_the_set_of_its_start(ctx, orc, form):
    torch = pytest.importorskip("torch")
    a, b = CUSTOM["long_below_short"], CUSTOM["short_wider"]
    reads = [synth.make_read(k, 9000, seed=31) for k in range(3)]
    signals = [orc.pa(*rd) for rd in reads]

    def entry(r, f, lo, hi):
        if form == "pa":
            return (r, f, signals[r][lo:hi])
        rd = reads[r]
        return (r, f, rd[0][lo:hi], rd[1], rd[2], rd[3])

    def push(entries, device):
        if device:
            return (device_push_pa if form == "pa" else device_push)(torch, ctx, entries, torch.cuda.current_stream())[0]
        return tables(ctx.live_push_pa(entries) if form == "pa" else ctx.live_push(entries))

    ctx.set_detector(sg.Detector(*a))
    t0 = push([entry(0, START, 0, 3000)], False)            # read 0 starts under A
    ctx.set_detector(sg.Detector(*b))
    t1 = push([entry(0, 0, 3000, 6000), entry(1, START, 0, 4000)], True)  # read 1 under B; read 0 keeps A
    ctx.set_detector(None)
    t2 = push([entry(0, END, 6000, 9000), entry(1, 0, 4000, 9000), entry(2, START, 0, 5000)], False)
    ctx.set_detector(sg.Detector(*a))
    t3 = push([entry(1, END, 9000, 9000), entry(2, END, 5000, 9000)], True)  # read 2 keeps the reference's set
    ref0, _ = stream_reference(orc, signals[0], 0, [3000, 3000, 3000], params=a)
    ref1, _ = stream_reference(orc, signals[1], 0, [4000, 5000, 0], params=b)
    ref2, _ = stream_reference(orc, signals[2], 0, [5000, 4000])
    for got, want in ((t0[0], ref0[0]), (t1[0], ref0[1]), (t2[0], ref0[2]), (t1[1], ref1[0]), (t2[1], ref1[1]),
                      (t3[0], ref1[2]), (t2[2], ref2[0]), (t3[1], ref2[1])):
        assert same_events(got, want)


@gpu
@pytest.mark.parametrize("form", ["int16", "pa"])
def test_live_dense_set_on_full_pushes(orc, form):
    """pushes that fill a slot, under the densest set, on a signal with an event every 3 samples: the staging grows
    and every entry reports what the streaming reference reports"""
    params = CUSTOM["dense"]
    n_ch, per = 32, (1 << 16) // 32 // (2 if form == "pa" else 1)
    pattern = np.array([10, 10, 20], np.int16)
    with sg.Context(device=0, max_samples=1 << 16, max_reads=n_ch) as c:
        c.live_open(n_ch)
        c.set_detector(sg.Detector(*params))
        reads = [(np.tile(np.roll(pattern, ch), 3 * per)[:3 * per], 8192.0, 4.0 + ch, 1400.0) for ch in range(n_ch)]
        signals = [orc.pa(*rd) for rd in reads]
        got = [[] for _ in range(n_ch)]
        for k in range(3):
            f = (START if k == 0 else 0) | (END if k == 2 else 0)
            if form == "pa":
                entries = [(ch, f, signals[ch][k * per:(k + 1) * per]) for ch in range(n_ch)]
                res = tables(c.live_push_pa(entries))
            else:
                entries = [(ch, f, reads[ch][0][k * per:(k + 1) * per], 8192.0, 4.0 + ch, 1400.0) for ch in range(n_ch)]
                res = tables(c.live_push(entries))
            assert c.counters()["status"] == 0
            for ch in range(n_ch):
                got[ch].append(res[ch])
        for ch in range(n_ch):
            ref, _ = stream_reference(orc, signals[ch], 0, [per] * 3, params=params)
            assert all(same_events(g, w) for g, w in zip(got[ch], ref)), ch
            assert len(concat(got[ch])[0]) >= per // 2

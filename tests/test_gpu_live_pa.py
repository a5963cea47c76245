"""Live event detection on the caller's pA floats (sgpu_slot_add_live_pa / sgpu_run_device_live_pa): every entry reports
what the streaming reference (tests/_live_ref.py) reports for that chunk, the entries of a read taken together equal the
pA batch path (sgpu_slot_add_read_pa) on the whole read, every float by its bits, and the pA of an int16 read streamed as
floats reports exactly what its int16 entries report. A read keeps the form of the entry that started it."""
import ctypes as C

import numpy as np
import pytest

from _live_ref import concat, same_events, split_lengths, stream_reference, whole_read
from _oracle import Oracle
from _oracle_pa import getevents_pa
from test_gpu_live import all_sources, device_push, schedule, stream, tables
from test_live_contract import late_long_peaks, long_read
import sigtk_b200 as sg
from sigtk_b200 import _lib, synth

gpu = pytest.mark.gpu

E_INVAL, E_FULL, E_TOOBIG, E_STATE = -1, -4, -5, -6
START, END, RNA = sg.LIVE_START, sg.LIVE_END, sg.LIVE_RNA


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 22, max_reads=1024) as c:
        c.live_open(1024)
        yield c


def normalised(rng, n):
    """z-normalised float noise around levels: sums that round in any order but the reference's"""
    x = synth.make_read(int(rng.integers(1 << 30)), n, seed=77)[0].astype(np.float32) * np.float32(0.17)
    x += rng.normal(0, 0.3, n).astype(np.float32)
    return ((x - np.float32(x.mean())) / np.float32(max(float(x.std()), 1e-3))).astype(np.float32)


def arbitrary_signals(seed):
    """floats the batch path's exactness witness refuses, and lengths around w2, 2 * w2 and the kernel's 256-sample
    tiles"""
    rng = np.random.default_rng(seed)
    out = [normalised(rng, int(n)) for n in rng.integers(200, 20000, 8)]
    out += [normalised(rng, n) for n in (1, 13, 27, 28, 29, 255, 256, 257, 511, 512, 513)]
    out.append(np.zeros(0, np.float32))
    out.append((normalised(rng, 3000) * np.float32(1e30)).astype(np.float32))
    out.append(np.full(2000, 1e30, np.float32))
    sub = (rng.integers(-40, 40, 3000) * np.float32(2.0 ** -149)).astype(np.float32)  # subnormal
    sub[::5] = 0.0
    out.append(sub)
    out.append((np.abs(normalised(rng, 2500)) * np.float32(1e-37)).astype(np.float32))  # near the smallest normal
    out += [np.full(n, v, np.float32) for n, v in ((3000, 87.5), (999, -3.25e-3), (600, 0.0))]
    wide = normalised(rng, 9000)
    wide[::50] *= np.float32(1e6)
    out.append(wide)
    return out


# ---- the premise: the streaming reference on arbitrary floats is the whole read's getevents ---------------------------
def test_stream_reference_on_arbitrary_floats(orc):
    """the streaming reference had only been run on the pA of int16 samples; on any finite floats its chunks, taken
    together, are getevents(n, pa, rna) of the whole read"""
    for rna in (0, 1):
        rng = np.random.default_rng(40 + rna)
        for r, pa in enumerate(arbitrary_signals(300 + rna)):
            want = getevents_pa(orc, pa, rna) if len(pa) else None
            for _ in range(3):
                chunks = split_lengths(len(pa), rng)
                got = concat(stream_reference(orc, pa, rna, chunks)[0])
                if want is None:
                    assert got[0].size == 0
                else:
                    assert same_events(got, want), f"rna={rna} signal {r} (n={len(pa)}) split {chunks[:8]}"


# ---- helpers -------------------------------------------------------------------------------------------------------
def schedule_pa(signals, rnas, rng, channels=None, splits=None):
    """the pushes that stream pA `signals` (one channel each) in seeded random splits, as test_gpu_live.schedule"""
    splits = splits or [split_lengths(len(s), rng) for s in signals]
    channels = channels or list(range(len(signals)))
    pushes = []
    for r, (s, rna, ch) in enumerate(zip(signals, rnas, channels)):
        at = 0
        for k, m in enumerate(splits[r]):
            f = (START | (RNA if rna else 0) if k == 0 else 0) | (END if k == len(splits[r]) - 1 else 0)
            while len(pushes) <= k:
                pushes.append([])
            pushes[k].append((r, k, (ch, f, s[at:at + m])))
            at += m
    return pushes, splits


def stream_pa(ctx, signals, rnas, rng, **kw):
    """-> the tables each signal's entries report, in order, and the splits"""
    pushes, splits = schedule_pa(signals, rnas, rng, **kw)
    out = [[None] * len(s) for s in splits]
    for push in pushes:
        for (r, k, _), t in zip(push, tables(ctx.live_push_pa([e for _, _, e in push]))):
            out[r][k] = t
    return out, splits


def batch_pa(ctx, signals, rnas):
    """the pA batch path's table of every whole signal, in batches that fit a slot"""
    out = [None] * len(signals)
    cap = ctx.max_samples // 2
    for rna in (0, 1):
        idx = [r for r in range(len(signals)) if rnas[r] == rna]
        while idx:
            group, used = [], 0
            while idx and (not group or used + (len(signals[idx[0]]) + 7) // 8 * 8 <= cap):
                used += (len(signals[idx[0]]) + 7) // 8 * 8
                group.append(idx.pop(0))
            res = ctx.run_pa([signals[r] for r in group], rna=rna)
            for j, r in enumerate(group):
                ev = res.events(j)
                out[r] = (ev.start, ev.length, ev.mean, ev.stdv)
    return out


def bits(a):
    a = np.asarray(a, np.float32)
    return a.view(np.uint32)


def same_floats(a, b):
    """bit-identical, except that a NaN only has to be a NaN"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(a[~na]), bits(b[~nb]))


def same_events_nan(a, b):
    return (np.array_equal(np.asarray(a[0], np.uint64), np.asarray(b[0], np.uint64)) and
            np.array_equal(bits(a[1]), bits(b[1])) and same_floats(a[2], b[2]) and same_floats(a[3], b[3]))


def check_signals(orc, signals, rnas, got, splits, batch=None, thr_long=None, same=same_events):
    for r, (pa, rna) in enumerate(zip(signals, rnas)):
        ref, _ = stream_reference(orc, pa, rna, splits[r], thr_long)
        for k in range(len(splits[r])):
            assert same(got[r][k], ref[k]), f"signal {r} (n={len(pa)}, rna={rna}) chunk {k} of {splits[r][:6]}"
        if batch is not None:
            assert same(concat(got[r]), batch[r]), f"signal {r} (n={len(pa)}, rna={rna}) vs the pA batch path"
        else:
            assert same(concat(got[r]), whole_read(orc, pa, rna, thr_long)), f"signal {r}"


def device_push_pa(torch, c, entries, stream):
    """sgpu_run_device_live_pa on device copies of `entries` (channel, flags, pa); -> their tables, the status"""
    lens = np.array([len(e[2]) for e in entries], np.int64)
    off = np.zeros(len(entries) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(max(int(off[-1]), 8), np.float32)
    for k, e in enumerate(entries):
        flat[off[k]:off[k] + lens[k]] = e[2]
    dev = torch.device("cuda:0")
    arrs = [torch.from_numpy(x).to(dev) for x in (flat, off, lens.astype(np.int32),
                                                   np.array([e[0] for e in entries], np.int32),
                                                   np.array([e[1] for e in entries], np.int32))]
    torch.cuda.synchronize()
    d = c.run_device_live_pa(*[a.data_ptr() for a in arrs], len(entries), int(off[-1]), stream.cuda_stream)
    torch.cuda.synchronize()
    cnt = c.counters()
    ne = cnt["n_events"]
    evs = sg.live_tables(c.d2h(d.ev_off, np.uint64, len(entries) + 1), c.d2h(d.ev_start, np.uint32, ne),
                         c.d2h(d.ev_len, np.uint32, ne), c.d2h(d.ev_mean, np.float32, ne),
                         c.d2h(d.ev_stdv, np.float32, ne))
    return tables(evs), cnt["status"]


# ---- parity ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_parity_on_the_pa_of_int16_reads(ctx, orc, seed):
    """the pA of the int16 live sources (synthetic reads, sp1_dna, synth_rna), DNA and RNA channels in the same pushes:
    every entry as the streaming reference, every read as the pA batch path, and every entry as the int16 entry of the
    same chunk of the same read"""
    reads, rnas = all_sources()
    signals = [orc.pa(*rd) for rd in reads]
    batch = batch_pa(ctx, signals, rnas)
    got, splits = stream_pa(ctx, signals, rnas, np.random.default_rng(seed))
    check_signals(orc, signals, rnas, got, splits, batch=batch)
    got16, _ = stream(ctx, reads, rnas, None, splits=splits)
    for r in range(len(reads)):
        for k in range(len(splits[r])):
            assert same_events(got[r][k], got16[r][k]), f"read {r} chunk {k}: pA entry vs int16 entry"


@gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_parity_on_arbitrary_floats(ctx, orc, seed):
    """signals whose sums the batch path must form in the reference's order (its witness fails), constants, values
    near 1e30 and near the subnormals, and lengths around w2 and the 256-sample tiles"""
    signals = arbitrary_signals(seed)
    rnas = [k % 2 for k in range(len(signals))]
    batch = batch_pa(ctx, signals, rnas)
    got, splits = stream_pa(ctx, signals, rnas, np.random.default_rng(100 + seed))
    check_signals(orc, signals, rnas, got, splits, batch=batch, same=same_events_nan)


@gpu
def test_nan_and_inf(ctx, orc):
    """NaN and Inf at chunk edges and inside the detector's windows: the boundaries of the batch path on the whole
    read, NaN statistics in the same places"""
    rng = np.random.default_rng(5)
    signals, splits = [], []
    for rna in (0, 1):
        for bad in (np.nan, np.inf, -np.inf):
            x = normalised(rng, 6000)
            sp = [100, 1, 13, 500, 2000, 6, 3380, 0]
            edges = np.cumsum(sp)[:-2]
            x[edges[0]] = bad              # the first sample of a chunk
            x[edges[2] - 1] = bad          # the last sample of a chunk
            x[edges[3] + 7] = bad          # inside a window, away from the edges
            x[4000] = bad
            signals.append(x)
            splits.append(sp)
        y = normalised(rng, 3000)
        y[1500] = np.nan
        y[2200] = np.inf
        signals.append(y)
        splits.append(split_lengths(3000, rng))
    rnas = [0] * 4 + [1] * 4
    batch = batch_pa(ctx, signals, rnas)
    got, _ = stream_pa(ctx, signals, rnas, None, splits=splits)
    check_signals(orc, signals, rnas, got, splits, batch=batch, same=same_events_nan)


@gpu
@pytest.mark.parametrize("push", [37, 2000])
def test_long_detector_across_pushes(ctx, orc, push):
    reads = [long_read(), long_read(), synth.make_read_cb(3, 9000)]
    rnas = [0, 1, 0]
    signals = [orc.pa(*rd) for rd in reads]
    splits = [[push] * (len(s) // push) + [len(s) % push] for s in signals]
    ctx.set_param(_lib.PARAM_THR_LONG, 1.0)
    try:
        got, _ = stream_pa(ctx, signals, rnas, None, splits=splits)
        got16, _ = stream(ctx, reads, rnas, None, splits=splits)
    finally:
        ctx.set_param(_lib.PARAM_THR_LONG, 9.0)
    check_signals(orc, signals, rnas, got, splits, thr_long=1.0)
    for r in range(len(reads)):
        assert same_events(concat(got[r]), concat(got16[r])), f"read {r}: pA vs int16 entries"
    if push == 37:
        assert late_long_peaks(orc, signals[0], 0, splits[0], 1.0)


@gpu
def test_long_reads(orc):
    """2,000,000-sample pA reads (DNA and RNA) in 2,000-sample pushes"""
    rng = np.random.default_rng(2000)
    signals = [normalised(rng, 2_000_000), orc.pa(*synth.make_read_cb(901, 2_000_000))]
    rnas = [0, 1]
    splits = [[2000] * 1000, [2000] * 1000]
    with sg.Context(device=0, max_samples=1 << 22, max_reads=64) as c:
        c.live_open(16)
        batch = batch_pa(c, signals, rnas)
        got, _ = stream_pa(c, signals, rnas, None, splits=splits, channels=[3, 11])
    check_signals(orc, signals, rnas, got, splits, batch=batch)


@gpu
def test_push_larger_than_the_grid(orc):
    """a push of 20,480 pA entries (more than the kernel's grid of warps), in three pushes per read"""
    n = 20480
    reads = [synth.make_read_cb(5000 + k, 150 + (k * 37) % 400) for k in range(n)]
    signals = [orc.pa(*rd) for rd in reads]
    rnas = [k % 3 == 0 for k in range(n)]
    splits = [[60, 40, len(s) - 100] for s in signals]
    with sg.Context(device=0, max_samples=1 << 24, max_reads=n) as c:
        c.live_open(n)
        got, _ = stream_pa(c, signals, rnas, None, splits=splits)
    for r in range(n):
        assert same_events(concat(got[r]), whole_read(orc, signals[r], int(rnas[r]))), f"read {r}"


# ---- both forms in one context -----------------------------------------------------------------------------------------
@gpu
def test_both_forms_on_two_slots_in_flight(ctx, orc):
    """int16 channels on slot 0 and pA channels on slot 1, both submitted before either is waited for, push by push"""
    reads = [synth.make_read_cb(180 + k, 3000 + 700 * k) for k in range(6)]
    rnas = [k % 2 for k in range(6)]
    signals = [orc.pa(*rd) for rd in reads]
    splits = [[1000, 1000, len(rd[0]) - 2000] for rd in reads]
    p16, _ = schedule(reads, rnas, None, channels=[600 + k for k in range(6)], splits=splits)
    ppa, _ = schedule_pa(signals, rnas, None, channels=[610 + k for k in range(6)], splits=splits)
    got16, gotpa = [[None] * 3 for _ in reads], [[None] * 3 for _ in reads]
    for p in range(3):
        ctx.live_fill(0, [e for _, _, e in p16[p]])
        ctx.live_fill_pa(1, [e for _, _, e in ppa[p]])
        ctx.submit(0, sg.WANT_EVENTS)
        ctx.submit(1, sg.WANT_EVENTS)
        for (r, k, _), t in zip(p16[p], tables(ctx.live_wait(0))):
            got16[r][k] = t
        for (r, k, _), t in zip(ppa[p], tables(ctx.live_wait(1))):
            gotpa[r][k] = t
    check_signals(orc, signals, rnas, gotpa, splits)
    for r in range(len(reads)):
        for k in range(3):
            assert same_events(got16[r][k], gotpa[r][k]), (r, k)


@gpu
def test_channel_reused_across_forms(ctx, orc):
    a, b, c = synth.make_read_cb(270, 5000), synth.make_read_cb(271, 4000), synth.make_read_cb(272, 3000)
    pa_a, pa_b, pa_c = orc.pa(*a), orc.pa(*b), orc.pa(*c)
    ch = 900
    # an int16 read ended, then a pA read on the channel
    t = tables(ctx.live_push([(ch, START, a[0][:2000], *a[1:])]))[0]
    t2 = tables(ctx.live_push([(ch, END, a[0][2000:], *a[1:])]))[0]
    assert same_events(concat([t, t2]), whole_read(orc, pa_a, 0))
    u = [tables(ctx.live_push_pa([(ch, START | RNA, pa_b[:1500])]))[0],
         tables(ctx.live_push_pa([(ch, END, pa_b[1500:])]))[0]]
    assert same_events(concat(u), whole_read(orc, pa_b, 1))
    # a pA read left open, discarded by an int16 START
    ctx.live_push_pa([(ch, START, pa_a[:2500])])
    v = [tables(ctx.live_push([(ch, START, c[0][:1000], *c[1:])]))[0],
         tables(ctx.live_push([(ch, 0, c[0][1000:2000], *c[1:])]))[0],
         tables(ctx.live_push([(ch, END, c[0][2000:], *c[1:])]))[0]]
    assert same_events(concat(v), whole_read(orc, pa_c, 0))
    # an int16 read left open, discarded by a pA START
    ctx.live_push([(ch, START | RNA, a[0][:2500], *a[1:])])
    w = [tables(ctx.live_push_pa([(ch, START, pa_c[:10])]))[0],
         tables(ctx.live_push_pa([(ch, 0, pa_c[10:2900])]))[0],
         tables(ctx.live_push_pa([(ch, END, pa_c[2900:])]))[0]]
    assert same_events(concat(w), whole_read(orc, pa_c, 0))


# ---- refusals ---------------------------------------------------------------------------------------------------------
@gpu
def test_form_mismatch_on_the_host_path(orc):
    """an entry that continues a read of the other form is refused by sgpu_submit, whatever its length and flags, and
    nothing of the push is queued; the reads are then finished correctly"""
    a, b = synth.make_read_cb(290, 3000), synth.make_read_cb(291, 2500)
    pa_a, pa_b = orc.pa(*a), orc.pa(*b)
    with sg.Context(device=0, max_samples=1 << 16, max_reads=64) as c:
        c.live_open(8)
        lib, h = c._lib, c._h
        head16 = tables(c.live_push([(0, START, a[0][:100], *a[1:])]))[0]   # channel 0: an int16 read
        headpa = tables(c.live_push_pa([(1, START, pa_b[:100])]))[0]       # channel 1: a pA read
        for flags, n in ((0, 10), (END, 10), (END, 0), (0, 0)):
            # a pA entry on channel 0, next to a START on channel 2 that must not happen
            c.live_fill_pa(0, [(2, START, pa_a[:50]), (0, flags, pa_a[100:100 + n])])
            assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE, (flags, n)
            c.live_fill(0, [(2, START, a[0][:50], *a[1:]), (1, flags, b[0][100:100 + n], *b[1:])])
            assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE, (flags, n)
        # channel 2 was never opened: samples without START are refused in either form
        c.live_fill_pa(0, [(2, 0, pa_a[:10])])
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
        t16 = tables(c.live_push([(0, END, a[0][100:], *a[1:])]))[0]
        tpa = tables(c.live_push_pa([(1, END, pa_b[100:])]))[0]
        assert same_events(concat([head16, t16]), whole_read(orc, pa_a, 0))
        assert same_events(concat([headpa, tpa]), whole_read(orc, pa_b, 0))


@gpu
def test_form_mismatch_on_the_device_path_and_the_mirror(orc):
    """sgpu_run_device_live(_pa) report a form mismatch as status and leave the channel as it was; the host mirror
    follows device-resident runs of both forms"""
    torch = pytest.importorskip("torch")
    a, b = synth.make_read_cb(390, 3000), synth.make_read_cb(391, 2500)
    pa_a, pa_b = orc.pa(*a), orc.pa(*b)
    s = torch.cuda.Stream()
    with sg.Context(device=0, max_samples=1 << 16, max_reads=64) as c:
        c.live_open(8)
        lib, h = c._lib, c._h
        g16, st = device_push(torch, c, [(0, START, a[0][:100], *a[1:])], s)       # channel 0: int16, on the device
        assert st == 0
        gpa, st = device_push_pa(torch, c, [(1, START, pa_b[:100])], s)             # channel 1: pA, on the device
        assert st == 0
        for flags, n in ((0, 10), (END, 0), (0, 0)):
            _, st = device_push_pa(torch, c, [(0, flags, pa_a[100:100 + n])], s)
            assert st == E_STATE, (flags, n)
            _, st = device_push(torch, c, [(1, flags, b[0][100:100 + n], *b[1:])], s)
            assert st == E_STATE, (flags, n)
        # the host mirror read back from the device: the forms are refused on the host path too
        c.live_fill_pa(0, [(0, 0, pa_a[100:110])])
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
        c.live_fill(0, [(1, END, b[0][100:100], *b[1:])])
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
        # and the right forms continue both reads, on the host path, then on the device
        m16 = tables(c.live_push([(0, 0, a[0][100:1000], *a[1:])]))[0]
        mpa = tables(c.live_push_pa([(1, 0, pa_b[100:1000])]))[0]
        e16, st = device_push(torch, c, [(0, END, a[0][1000:], *a[1:])], s)
        assert st == 0
        epa, st = device_push_pa(torch, c, [(1, END, pa_b[1000:])], s)
        assert st == 0
        assert same_events(concat([g16[0], m16, e16[0]]), whole_read(orc, pa_a, 0))
        assert same_events(concat([gpa[0], mpa, epa[0]]), whole_read(orc, pa_b, 0))
        # both closed now, as the mirror knows after the device runs
        c.live_fill_pa(0, [(0, 0, pa_a[:10])])
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
        # the device path's other refusals
        for entries, code in (([(3, START | 16, pa_a[:50])], E_INVAL),        # unknown flag
                              ([(8, START, pa_a[:50])], E_INVAL),             # channel >= n_channels
                              ([(4, START, pa_a[:50]), (4, 0, pa_a[:50])], E_INVAL)):  # one channel twice
            _, st = device_push_pa(torch, c, entries, s)
            assert st == code, entries
        got, st = device_push_pa(torch, c, [(5, START | END, pa_a)], s)
        assert st == 0 and same_events(got[0], whole_read(orc, pa_a, 0))


MAX_SAMPLES, MAX_READS, N_CHANNELS = 4096, 8, 8
RAW = np.random.default_rng(3).normal(500, 60, 100).astype(np.int16)
PA = np.linspace(60.0, 90.0, 100).astype(np.float32)
OTHERS = ("none", "int16", "svbzd", "pa", "live")


@pytest.fixture(scope="module")
def small():
    with sg.Context(device=0, max_samples=MAX_SAMPLES, max_reads=MAX_READS) as c:
        c.live_open(N_CHANNELS)
        yield c, Oracle().svbzd_encode(RAW)


def add(c, svb, kind, slot=0, channel=0):
    """appends one small record of `kind` (each live entry a whole read); -> the return code"""
    lib, h = c._lib, c._h
    if kind == "live_pa":
        return lib.sgpu_slot_add_live_pa(h, slot, channel, START | END, PA.ctypes.data, PA.size)
    if kind == "int16":
        return lib.sgpu_slot_add_read(h, slot, RAW.ctypes.data, RAW.size, 8192.0, 4.0, 1400.0)
    if kind == "svbzd":
        return lib.sgpu_slot_add_read_svbzd(h, slot, svb.ctypes.data, svb.size, 8192.0, 4.0, 1400.0)
    if kind == "pa":
        return lib.sgpu_slot_add_read_pa(h, slot, PA.ctypes.data, PA.size)
    assert kind == "live"
    return lib.sgpu_slot_add_live(h, slot, channel, START | END, RAW.ctypes.data, RAW.size, 8192.0, 4.0, 1400.0)


def fill(c, svb, kind, slot=0):
    assert c._lib.sgpu_slot_reset(c._h, slot, 0) == 0
    if kind != "none":
        assert add(c, svb, kind, slot) == 0


def wait(c, kind, slot=0):
    if kind in ("live", "live_pa"):
        return c._lib.sgpu_wait_live(c._h, slot, C.byref(_lib.LiveResult()))
    return c._lib.sgpu_wait(c._h, slot, C.byref(_lib.Result()))


@gpu
@pytest.mark.parametrize("other", OTHERS)
def test_one_kind_per_slot(small, other):
    c, svb = small
    for first, second in (("live_pa", other), (other, "live_pa")):
        fill(c, svb, first)
        if second != "none":   # (an empty slot takes every kind; a slot of live_pa entries takes no other)
            assert add(c, svb, second, channel=1) == (0 if first == "none" else E_STATE), (first, second)
        assert c._lib.sgpu_slot_reset(c._h, 0, 0) == 0
        if second != "none":
            assert add(c, svb, second) == 0, (first, second)   # a reset slot takes every kind
    assert c._lib.sgpu_slot_reset(c._h, 0, 0) == 0


@gpu
def test_submitted_slot_and_wants(small):
    c, svb = small
    lib, h = c._lib, c._h
    fill(c, svb, "live_pa")
    assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == 0
    for other in OTHERS[1:] + ("live_pa",):
        assert add(c, svb, other, channel=2) == E_STATE, other
    assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
    assert lib.sgpu_slot_reset(h, 0, 0) == E_STATE
    assert lib.sgpu_wait(h, 0, C.byref(_lib.Result())) == E_STATE        # sgpu_wait refuses a live slot
    assert wait(c, "live_pa") == 0
    assert wait(c, "live_pa") == E_STATE
    for want in range(64):
        fill(c, svb, "live_pa")
        rc = lib.sgpu_submit(h, 0, want)
        if want == sg.WANT_EVENTS:
            assert rc == 0
            assert wait(c, "live_pa") == 0
        else:
            assert rc == E_INVAL, want
            assert wait(c, "live_pa") == E_STATE, want
    fill(c, svb, "pa")                                                    # and sgpu_wait_live refuses the others
    assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == 0
    assert lib.sgpu_wait_live(h, 0, C.byref(_lib.LiveResult())) == E_STATE
    assert wait(c, "pa") == 0


@gpu
def test_append_checks_and_capacity(small):
    c, _ = small
    lib, h = c._lib, c._h
    bigf = np.zeros(MAX_SAMPLES, np.float32)

    def live(n, channel=0, flags=START):
        return lib.sgpu_slot_add_live_pa(h, 0, channel, flags, bigf.ctypes.data, n)

    # max_samples / 2 floats, every entry padded to 8; 2^31 samples never
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    assert live(MAX_SAMPLES // 2 + 1) == E_TOOBIG
    assert live(1 << 31) == E_TOOBIG
    assert live((1 << 31) - 1) == E_TOOBIG
    assert live(MAX_SAMPLES // 2 - 7) == 0
    assert live(1, 1) == E_FULL
    assert live(MAX_SAMPLES // 2 + 1, 1) == E_TOOBIG
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    for r in range(MAX_READS):
        assert live(0, r % N_CHANNELS) == r
    assert live(0, 0) == E_FULL
    # the channel and the flags before the length, the second entry of a channel after it
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    assert live(1 << 31, N_CHANNELS) == E_INVAL
    assert live(1 << 31, 0, START | 8) == E_INVAL
    assert live(MAX_SAMPLES // 2 - 8, 0) == 0
    assert live(16, 0) == E_FULL
    assert live(MAX_SAMPLES, 0) == E_TOOBIG
    assert live(0, 0) == E_INVAL
    assert live(0, 1) == 1
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    assert lib.sgpu_slot_add_live_pa(h, 0, 0, START, None, 4) == E_INVAL
    assert lib.sgpu_slot_add_live_pa(None, 0, 0, START, bigf.ctypes.data, 4) == E_INVAL


@gpu
def test_before_live_open_and_device_batch_limits():
    torch = pytest.importorskip("torch")
    x = np.zeros(64, np.float32)
    with sg.Context(device=0, max_samples=1024, max_reads=4) as c:
        lib, h = c._lib, c._h
        assert lib.sgpu_slot_reset(h, 0, 0) == 0
        assert lib.sgpu_slot_add_live_pa(h, 0, 0, START, x.ctypes.data, 64) == E_STATE
        with pytest.raises(sg.SgpuError) as e:
            c.run_device_live_pa(0, 0, 0, 0, 0, 0, 0)
        assert e.value.code == E_STATE
        c.live_open(8)
        dev = torch.device("cuda:0")
        pa = torch.zeros(2048, dtype=torch.float32, device=dev)
        off = torch.zeros(6, dtype=torch.int64, device=dev)
        ln = torch.zeros(5, dtype=torch.int32, device=dev)
        ch = torch.arange(5, dtype=torch.int32, device=dev)
        fl = torch.full((5,), START, dtype=torch.int32, device=dev)
        ptrs = [t.data_ptr() for t in (pa, off, ln, ch, fl)]
        for n, span in ((1, 1025), (5, 0)):    # span > max_samples, n_entries > max_reads
            with pytest.raises(sg.SgpuError) as e:
                c.run_device_live_pa(*ptrs, n, span)
            assert e.value.code == E_INVAL, (n, span)
        with pytest.raises(sg.SgpuError) as e:
            c.run_device_live_pa(0, *ptrs[1:], 1, 8)   # no floats
        assert e.value.code == E_INVAL
        c.run_device_live_pa(*ptrs, 4, 0)           # four empty START entries: nothing to refuse
        assert c.counters()["status"] == 0


# ---- device path ------------------------------------------------------------------------------------------------------
@gpu
def test_device_path_on_a_torch_stream(ctx, orc):
    torch = pytest.importorskip("torch")
    reads, rnas = all_sources()
    signals = [orc.pa(*rd) for rd in reads[:30]] + arbitrary_signals(7)
    rnas = rnas[:30] + [k % 2 for k in range(len(signals) - 30)]
    pushes, _ = schedule_pa(signals, rnas, np.random.default_rng(19), channels=[300 + r for r in range(len(signals))])
    s = torch.cuda.Stream()
    with sg.Context(device=0, max_samples=1 << 22, max_reads=1024, flags=sg.F_NO_HOST_SLOTS) as c:
        c.live_open(1024)
        for push in pushes:
            entries = [e for _, _, e in push]
            host = tables(ctx.live_push_pa(entries))
            got, status = device_push_pa(torch, c, entries, s)
            assert status == 0
            for x, y in zip(host, got):
                assert same_events(x, y)

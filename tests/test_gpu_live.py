"""Live event detection on the GPU (sgpu_slot_add_live / sgpu_wait_live / sgpu_run_device_live, live.cu): the events
every entry reports equal the streaming reference's (tests/_live_ref.py) for that chunk, and the events of a read's
entries taken together equal both the int16 batch path on the whole read and the oracle, every float by its bits."""
import ctypes as C

import numpy as np
import pytest

from _live_ref import concat, same_events, split_lengths, stream_reference, whole_read
from _oracle import Oracle
from test_live_contract import golden, late_long_peaks, long_read
import sigtk_b200 as sg
from sigtk_b200 import _lib, synth

pytestmark = pytest.mark.gpu

E_INVAL, E_TOOBIG, E_STATE = -1, -5, -6
START, END, RNA = sg.LIVE_START, sg.LIVE_END, sg.LIVE_RNA


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def tables(evs):
    return [(t.start, t.length, t.mean, t.stdv) for t in evs]


def schedule(reads, rnas, rng, channels=None, splits=None):
    """the pushes that stream `reads` (one channel each) in seeded random splits: push p holds chunk p of every read
    that has one. -> (pushes: lists of (read, chunk, entry)), the splits"""
    splits = splits or [split_lengths(len(rd[0]), rng) for rd in reads]
    channels = channels or list(range(len(reads)))
    pushes = []
    for r, (rd, rna, ch) in enumerate(zip(reads, rnas, channels)):
        at = 0
        for k, m in enumerate(splits[r]):
            f = (START | (RNA if rna else 0) if k == 0 else 0) | (END if k == len(splits[r]) - 1 else 0)
            while len(pushes) <= k:
                pushes.append([])
            pushes[k].append((r, k, (ch, f, rd[0][at:at + m], rd[1], rd[2], rd[3])))
            at += m
    return pushes, splits


def stream(ctx, reads, rnas, rng, **kw):
    """-> the tables each read's entries report, in order, and the splits"""
    pushes, splits = schedule(reads, rnas, rng, **kw)
    out = [[None] * len(s) for s in splits]
    for push in pushes:
        got = ctx.live_push([e for _, _, e in push])
        for (r, k, _), t in zip(push, tables(got)):
            out[r][k] = t
    return out, splits


def check_reads(orc, reads, rnas, got, splits, thr_long=None, batch=None):
    for r, (rd, rna) in enumerate(zip(reads, rnas)):
        pa = orc.pa(*rd)
        ref, _ = stream_reference(orc, pa, rna, splits[r], thr_long)
        for k in range(len(splits[r])):
            assert same_events(got[r][k], ref[k]), f"read {r} (n={len(pa)}, rna={rna}) chunk {k} of {splits[r][:6]}"
        assert same_events(concat(got[r]), whole_read(orc, pa, rna, thr_long)), f"read {r}"
        if batch is not None:
            ev = batch[r]
            assert same_events(concat(got[r]), (ev.start, ev.length, ev.mean, ev.stdv)), f"read {r} vs ctx.run"


def batch_events(ctx, reads, rnas):
    out = [None] * len(reads)
    for rna in (0, 1):
        idx = [r for r in range(len(reads)) if rnas[r] == rna]
        if idx:
            res = ctx.run([reads[r] for r in idx], rna=rna)
            for j, r in enumerate(idx):
                out[r] = res.events(j)
    return out


def all_sources():
    cb = [synth.make_read_cb(k, n) for k, n in enumerate((0, 1, 5, 13, 27, 28, 29, 600, 7000, 20000, 61000))]
    reads = cb + cb + golden("sp1_dna.npz") + golden("synth_rna.npz")
    rnas = [0] * len(cb) + [1] * len(cb) + [0] * 100 + [1] * 12
    return reads, rnas


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 22, max_reads=1024) as c:
        c.live_open(1024)
        yield c


def test_parity_and_timing_of_reports(ctx, orc):
    """every read of the four sources, DNA and RNA channels with different calibrations in the same pushes; three
    split seeds give the same concatenations"""
    reads, rnas = all_sources()
    batch = batch_events(ctx, reads, rnas)
    first = None
    for seed in (1, 2, 3):
        got, splits = stream(ctx, reads, rnas, np.random.default_rng(seed))
        check_reads(orc, reads, rnas, got, splits, batch=batch)
        cat = [concat(g) for g in got]
        if first is None:
            first = cat
        assert all(same_events(a, b) for a, b in zip(cat, first))


@pytest.mark.parametrize("push", [37, 2000])
def test_long_detector_across_pushes(ctx, orc, push):
    reads = [long_read(), long_read(), synth.make_read_cb(3, 9000)]
    rnas = [0, 1, 0]
    splits = [[push] * (len(rd[0]) // push) + [len(rd[0]) % push] for rd in reads]
    ctx.set_param(_lib.PARAM_THR_LONG, 1.0)
    try:
        got, _ = stream(ctx, reads, rnas, None, splits=splits)
    finally:
        ctx.set_param(_lib.PARAM_THR_LONG, 9.0)
    check_reads(orc, reads, rnas, got, splits, thr_long=1.0)
    if push == 37:
        pa = orc.pa(*reads[0])
        assert late_long_peaks(orc, pa, 0, splits[0], 1.0) and late_long_peaks(orc, pa, 1, splits[1], 1.0)


def test_long_reads(orc):
    """2,000,000-sample reads in 2,000-sample pushes, next to short reads that open and close on other channels"""
    longs = [synth.make_read_cb(900, 2_000_000), synth.make_read_cb(901, 2_000_000)]
    shorts = [synth.make_read_cb(1000 + k, 3000 + 997 * k) for k in range(40)]
    reads = longs + shorts
    rnas = [0, 1] + [k % 2 for k in range(40)]
    splits = [[2000] * 1000, [2000] * 1000] + [[1000] * (len(rd[0]) // 1000) + [len(rd[0]) % 1000] for rd in shorts]
    # the short reads take turns on channels 2..9: a read starts on its channel once the previous one has ended
    with sg.Context(device=0, max_samples=1 << 22, max_reads=64) as c:
        c.live_open(16)
        batch = batch_events(c, reads, rnas)
        out = [[None] * len(s) for s in splits]
        queue = {ch: [r for r in range(2, len(reads)) if 2 + (r - 2) % 8 == ch] for ch in range(2, 10)}
        cur = {ch: (q.pop(0), 0) for ch, q in queue.items()}
        at = [0] * len(reads)
        for p in range(1000):
            entries, who = [], []
            for r in (0, 1):
                f = (START | (RNA if rnas[r] else 0) if p == 0 else 0) | (END if p == 999 else 0)
                entries.append((r, f, reads[r][0][at[r]:at[r] + 2000], *reads[r][1:]))
                who.append((r, p))
                at[r] += 2000
            for ch in range(2, 10):
                if cur.get(ch) is None:
                    continue
                r, k = cur[ch]
                m = splits[r][k]
                f = (START | (RNA if rnas[r] else 0) if k == 0 else 0) | (END if k == len(splits[r]) - 1 else 0)
                entries.append((ch, f, reads[r][0][at[r]:at[r] + m], *reads[r][1:]))
                who.append((r, k))
                at[r] += m
                cur[ch] = (r, k + 1) if k + 1 < len(splits[r]) else ((queue[ch].pop(0), 0) if queue[ch] else None)
            for (r, k), t in zip(who, tables(c.live_push(entries))):
                out[r][k] = t
        assert all(v is None for v in cur.values())
        check_reads(orc, reads, rnas, out, splits, batch=batch)


def test_push_larger_than_the_grid(orc):
    """a push of 20,480 entries (more than the kernel's grid of warps), in three pushes per read"""
    n = 20480
    reads = [synth.make_read_cb(5000 + k, 150 + (k * 37) % 400) for k in range(n)]
    rnas = [k % 3 == 0 for k in range(n)]
    splits = [[60, 40, len(rd[0]) - 100] for rd in reads]
    with sg.Context(device=0, max_samples=1 << 24, max_reads=n) as c:
        c.live_open(n)
        got, _ = stream(c, reads, rnas, None, splits=splits)
    for r in range(n):
        pa = orc.pa(*reads[r])
        assert same_events(concat(got[r]), whole_read(orc, pa, int(rnas[r]))), f"read {r}"


def test_channel_reuse(ctx, orc):
    a, b, c = synth.make_read_cb(70, 5000), synth.make_read_cb(71, 4000), synth.make_read_cb(72, 3000)
    ch = 700
    # a new read after END
    t1 = tables(ctx.live_push([(ch, START | END, a[0], *a[1:])]))[0]
    t2 = tables(ctx.live_push([(ch, START, b[0][:1500], *b[1:])]))[0]
    t3 = tables(ctx.live_push([(ch, END, b[0][1500:], *b[1:])]))[0]
    assert same_events(t1, whole_read(orc, orc.pa(*a), 0))
    assert same_events(concat([t2, t3]), whole_read(orc, orc.pa(*b), 0))
    # START on an open channel discards the open read
    ctx.live_push([(ch, START, a[0][:2500], *a[1:])])
    u1 = tables(ctx.live_push([(ch, START | RNA, c[0][:1000], *c[1:])]))[0]
    u2 = tables(ctx.live_push([(ch, 0, c[0][1000:2000], *c[1:])]))[0]
    u3 = tables(ctx.live_push([(ch, END, c[0][2000:], *c[1:])]))[0]
    assert same_events(concat([u1, u2, u3]), whole_read(orc, orc.pa(*c), 1))


def test_two_slots_in_flight(ctx, orc):
    reads = [synth.make_read_cb(80 + k, 3000 + 500 * k) for k in range(6)]
    rnas = [k % 2 for k in range(6)]
    splits = [[1000, 1000, len(rd[0]) - 2000] for rd in reads]
    pushes, _ = schedule(reads, rnas, None, channels=[800 + k for k in range(6)], splits=splits)
    seq = [tables(ctx.live_push([e for _, _, e in p])) for p in pushes]
    pushes2, _ = schedule(reads, rnas, None, channels=[810 + k for k in range(6)], splits=splits)
    ctx.live_fill(0, [e for _, _, e in pushes2[0]])
    ctx.live_fill(1, [e for _, _, e in pushes2[1]])
    ctx.submit(0, sg.WANT_EVENTS)
    ctx.submit(1, sg.WANT_EVENTS)
    got = [tables(ctx.live_wait(0)), tables(ctx.live_wait(1))]
    got.append(tables(ctx.live_push([e for _, _, e in pushes2[2]])))
    for p in range(3):
        for x, y in zip(seq[p], got[p]):
            assert same_events(x, y)


def device_push(torch, c, entries, stream):
    """sgpu_run_device_live on device copies of `entries`; -> their tables"""
    lens = np.array([len(e[2]) for e in entries], np.int64)
    off = np.zeros(len(entries) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(max(int(off[-1]), 8), np.int16)
    for k, e in enumerate(entries):
        flat[off[k]:off[k] + lens[k]] = e[2]
    offf = np.array([np.float32(e[4]) for e in entries], np.float32)
    unit = np.array([np.float32(e[5]) / np.float32(e[3]) for e in entries], np.float32)
    dev = torch.device("cuda:0")
    arrs = [torch.from_numpy(x).to(dev) for x in (flat, off, lens.astype(np.int32),
                                                   np.array([e[0] for e in entries], np.int32),
                                                   np.array([e[1] for e in entries], np.int32), offf, unit)]
    torch.cuda.synchronize()
    d = c.run_device_live(*[a.data_ptr() for a in arrs], len(entries), int(off[-1]), stream.cuda_stream)
    torch.cuda.synchronize()
    cnt = c.counters()
    ne = cnt["n_events"]
    evs = sg.api.live_tables(c.d2h(d.ev_off, np.uint64, len(entries) + 1), c.d2h(d.ev_start, np.uint32, ne),
                             c.d2h(d.ev_len, np.uint32, ne), c.d2h(d.ev_mean, np.float32, ne),
                             c.d2h(d.ev_stdv, np.float32, ne))
    return tables(evs), cnt["status"]


def test_device_path_on_a_torch_stream(ctx, orc):
    torch = pytest.importorskip("torch")
    reads, rnas = all_sources()
    reads, rnas = reads[:40], rnas[:40]
    pushes, splits = schedule(reads, rnas, np.random.default_rng(9), channels=[100 + r for r in range(40)])
    s = torch.cuda.Stream()
    with sg.Context(device=0, max_samples=1 << 22, max_reads=1024, flags=sg.F_NO_HOST_SLOTS) as c:
        c.live_open(1024)
        for push in pushes:
            entries = [e for _, _, e in push]
            host = tables(ctx.live_push(entries))
            got, status = device_push(torch, c, entries, s)
            assert status == 0
            for x, y in zip(host, got):
                assert same_events(x, y)


def test_errors(orc):
    a, b = synth.make_read_cb(90, 3000), synth.make_read_cb(91, 2500)
    with sg.Context(device=0, max_samples=1 << 16, max_reads=64) as c:
        lib, h = c._lib, c._h
        raw = a[0]

        def add(slot, ch, f, x=raw[:100]):
            return lib.sgpu_slot_add_live(h, slot, ch, f, x.ctypes.data, len(x), a[1], a[2], a[3])
        assert add(0, 0, START) == E_STATE                     # before sgpu_live_open
        c.live_open(8)
        assert lib.sgpu_live_open(h, 8) == E_STATE
        lib.sgpu_slot_reset(h, 0, 0)
        assert add(0, 8, START) == E_INVAL                     # channel >= n_channels
        assert add(0, 0, START | 8) == E_INVAL                 # unknown flag
        assert add(0, 0, START) == 0
        assert add(0, 0, 0) == E_INVAL                         # a second entry for the channel
        assert lib.sgpu_slot_add_read(h, 0, raw.ctypes.data, 10, 8192.0, 0.0, 1.0) == E_STATE
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS | sg.WANT_PA) == E_INVAL
        assert c._lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == 0
        assert lib.sgpu_wait(h, 0, C.byref(_lib.Result())) == E_STATE
        head = tables(c.live_wait(0))[0]                       # channel 0: a[:100]
        big = np.zeros((1 << 16) + 8, np.int16)
        lib.sgpu_slot_reset(h, 0, 0)
        assert add(0, 1, START, big) == E_TOOBIG
        c.fill(1, [a], 0)
        assert add(1, 1, START) == E_STATE                     # an int16 slot
        c.submit(1, sg.WANT_EVENTS)
        assert lib.sgpu_wait_live(h, 1, C.byref(_lib.LiveResult())) == E_STATE
        c.wait(1, sg.WANT_EVENTS)
        # refused submits change no channel: channel 0 holds a[:100], channel 1 gets b's first chunk
        for entries, code in (([(1, START, b[0][:1000], *b[1:]), (5, 0, raw[:10], *a[1:])], E_STATE),
                              ([(1, START, b[0][:1000], *b[1:]), (6, END, raw[:0], *a[1:])], E_STATE)):
            c.live_fill(0, entries)
            assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == code
        t0 = tables(c.live_push([(0, 0, raw[100:2000], *a[1:]), (1, START, b[0][:1000], *b[1:])]))
        t1 = tables(c.live_push([(0, END, raw[2000:], *a[1:]), (1, END, b[0][1000:], *b[1:])]))
        first = tables(c.live_push([(2, START, raw[:0], *a[1:])]))  # (a read of channel 2 with no samples yet)
        assert first[0][0].size == 0
        assert same_events(concat([head, t0[0], t1[0]]), whole_read(orc, orc.pa(*a), 0))
        assert same_events(concat([t0[1], t1[1]]), whole_read(orc, orc.pa(*b), 0))
        # the device form reports the same violations as status and leaves the channels as they were
        torch = pytest.importorskip("torch")
        s = torch.cuda.Stream()
        for entries, code in (([(3, 0, raw[:50], *a[1:])], E_STATE),             # samples on a closed channel
                              ([(3, START | 16, raw[:50], *a[1:])], E_INVAL),     # unknown flag
                              ([(9, START, raw[:50], *a[1:])], E_INVAL),          # channel >= n_channels
                              ([(2, 0, raw[:50], *a[1:]), (2, 0, raw[:50], *a[1:])], E_INVAL)):  # one channel twice
            got, status = device_push(torch, c, entries, s)
            assert status == code, entries
        # channel 2: at most one of the two duplicate entries went through; finish from the device's own state
        got, status = device_push(torch, c, [(4, START | END, raw, *a[1:])], s)
        assert status == 0 and same_events(got[0], whole_read(orc, orc.pa(*a), 0))
        # the host mirror follows the device-resident runs: channel 3 is still closed
        c.live_fill(0, [(3, 0, raw[:10], *a[1:])])
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE

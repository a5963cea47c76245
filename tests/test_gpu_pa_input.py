"""Event detection on the caller's own pA floats: sgpu_slot_add_read_pa / sgpu_run_device_pa (pa_input.cu) against the
oracle's getevents(n, pa, rna) (orc_getevents) and against the int16 path.

Boundaries and the bits of every mean / stdv must match for finite input; with NaN or Inf in the input the boundaries
must match and the NaN statistics be NaN in the same places. seq_order[r] = 1 marks the reads whose prefix sums were
formed in the reference's order because the exactness witness failed (test_pa_witness.py restates the witness)."""
import os

import numpy as np
import pytest

import _fmt
from _oracle import Oracle
from _oracle_pa import getevents_pa
import sigtk_b200 as sg
from sigtk_b200 import synth
from test_pa_witness import witness
from test_gpu_waves import premise, single_pass, span_of, pmap

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_INVAL, E_STATE = -1, -6


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def sm(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 24, max_reads=8192) as c:
        yield c


def bits(a):
    a = np.asarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def same_floats(a, b):
    """bit-identical, except that a NaN only has to be a NaN"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(a[~na]), bits(b[~nb]))


def event_mismatch(ev, want, n):
    """what differs between an EventTable and the oracle's (start, length, mean, stdv); '' when nothing"""
    if n == 0:      # DESIGN §3 point 5: an empty record has no event (the oracle returns one of length 0)
        return "" if ev.n == 0 else "events of an empty record"
    st, ln, mn, sd = want
    if not np.array_equal(ev.start, st):
        return "event starts"
    if not (np.array_equal(bits(ev.length), bits(ln)) and same_floats(ev.mean, mn) and same_floats(ev.stdv, sd)):
        return "event length / mean / stdv"
    return ""


def check_oracle(orc, res, signals, rna):
    def one(r):
        return r, event_mismatch(res.events(r), getevents_pa(orc, signals[r], rna), len(signals[r]))
    bad = [(r, len(signals[r]), w) for r, w in pmap(one, range(len(signals))) if w]
    assert not bad, f"{len(bad)} of {len(signals)} reads differ (read, length, what): {bad[:8]}"


def assert_same_events(a, b):
    assert np.array_equal(a.ev_off, b.ev_off) and np.array_equal(a.ev_start, b.ev_start)
    assert same_floats(a.ev_mean, b.ev_mean) and same_floats(a.ev_stdv, b.ev_stdv)


def layout(signals):
    lens = np.array([len(s) for s in signals], np.int64)
    off = np.zeros(len(signals) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(max(int(off[-1]), 8), np.float32)
    for r, s in enumerate(signals):
        flat[off[r]:off[r] + lens[r]] = s
    return flat, off, lens


def run_device(torch, ctx, signals, rna, stream=None):
    """sgpu_run_device_pa on device copies of `signals`; -> a BatchResult with the event outputs"""
    flat, off, lens = layout(signals)
    dev = torch.device("cuda:0")
    d_pa, d_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    torch.cuda.synchronize()
    st = (stream or torch.cuda.current_stream()).cuda_stream
    d = ctx.run_device_pa(d_pa.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), len(signals), int(off[-1]), rna,
                          sg.WANT_EVENTS, st)
    torch.cuda.synchronize()
    c = ctx.counters()
    assert c["status"] == 0
    n, ne = len(signals), c["n_events"]
    res = sg.BatchResult(n_reads=n, read_len=lens.astype(np.uint32))
    res.ev_off = ctx.d2h(d.ev_off, np.uint64, n + 1)
    res.ev_start = ctx.d2h(d.ev_start, np.uint32, ne)
    res.ev_mean = ctx.d2h(d.ev_mean, np.float32, ne)
    res.ev_stdv = ctx.d2h(d.ev_stdv, np.float32, ne)
    res.seq_order = ctx.d2h(d.seq_order, np.uint32, n)
    res.fixups = ctx.d2h(d.fixups, np.uint32, n)
    assert not d.pa and not d.stat
    return res


# ---- round trip: the library's own pA fed back in ---------------------------------------------------------------------
@pytest.mark.parametrize("name,rna", [("sp1_dna.npz", 0), ("synth_rna.npz", 1)])
def test_round_trip_golden(torch, ctx, orc, name, rna):
    reads = [rd for _, rd in _fmt.load_npz(os.path.join(G, name))]
    raw = ctx.run(reads, rna=rna, want=sg.WANT_EVENTS | sg.WANT_PA)
    pa = [p.copy() for p in raw.pa]
    host = ctx.run_pa(pa, rna=rna)
    dev = run_device(torch, ctx, pa, rna)
    assert_same_events(host, raw)
    assert_same_events(dev, raw)
    assert np.array_equal(host.seq_order, dev.seq_order)
    check_oracle(orc, host, pa, rna)


def test_round_trip_past_the_grid(torch, orc, sm):
    """45,000 reads (tiny to 60 k samples): every new kernel's grid-stride loop comes round more than once; the same
    batch with every read summed in the reference's order (SGPU_F_FORCE_GENERIC) gives the same events"""
    cap = single_pass(sm)
    rng = np.random.default_rng(4545)
    lens = rng.integers(1, 1200, 45000)
    lens[::900] = rng.integers(20000, 60000, lens[::900].shape)
    reads = [synth.make_read(k, int(n), seed=4545) for k, n in enumerate(lens)]
    span = span_of(reads)
    tiles = int(((lens + 4095) // 4096).sum())
    premise("reads over pa_init_kernel's threads", len(reads), sm * 256, 1.1)
    premise("tiles over pa_tile_kernel / pa_scan_kernel's CTAs", tiles, sm * 8, 2.0)
    premise("reads over pa_read_kernel's warps", len(reads), sm * 8 * 4, 2.0)
    premise("reads over the warps of gen_prefix_pa / gen_detect_pa / gen_emit", len(reads), cap["gen_warp_reads"], 2.0)
    premise("reads over gen_tstat_kernel's CTAs", len(reads), cap["gen_tstat_reads"], 2.0)
    for rna in (0, 1):
        with sg.Context(device=0, max_samples=1 << 26, max_reads=65536, flags=sg.F_NO_HOST_SLOTS) as c:
            flat, off, lens_ = layout([rd[0] for rd in reads])
            # the int16 run from device memory, its pA read back
            dev = torch.device("cuda:0")
            raw16 = np.zeros(flat.shape[0], np.int16)
            for r, rd in enumerate(reads):
                raw16[off[r]:off[r] + lens_[r]] = rd[0]
            d_s, d_off = torch.from_numpy(raw16).to(dev), torch.from_numpy(off).to(dev)
            d_len = torch.from_numpy(lens_.astype(np.int32)).to(dev)
            d_o = torch.tensor([np.float32(rd[2]) for rd in reads], dtype=torch.float32, device=dev)
            d_u = torch.tensor([np.float32(np.float32(rd[3]) / np.float32(rd[1])) for rd in reads], dtype=torch.float32,
                               device=dev)
            torch.cuda.synchronize()
            d = c.run_device(d_s.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_o.data_ptr(), d_u.data_ptr(),
                             len(reads), span, rna, sg.WANT_EVENTS | sg.WANT_PA, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            ne = c.counters()["n_events"]
            pa_flat = c.d2h(d.pa, np.float32, span)
            ev16 = (c.d2h(d.ev_off, np.uint64, len(reads) + 1), c.d2h(d.ev_start, np.uint32, ne),
                    c.d2h(d.ev_mean, np.float32, ne), c.d2h(d.ev_stdv, np.float32, ne))
            pa = [pa_flat[off[r]:off[r] + lens_[r]].copy() for r in range(len(reads))]
            res = run_device(torch, c, pa, rna)
        assert np.array_equal(res.ev_off, ev16[0]) and np.array_equal(res.ev_start, ev16[1])
        assert np.array_equal(bits(res.ev_mean), bits(ev16[2])) and np.array_equal(bits(res.ev_stdv), bits(ev16[3]))
        n_seq = int(res.seq_order.sum())
        print(f"rna={rna}: {len(reads)} reads, {span} samples, {tiles} tiles, {n_seq} in the reference's order")
        assert n_seq <= len(reads) // 100
        check_oracle(orc, res, pa, rna)
        with sg.Context(device=0, max_samples=1 << 26, max_reads=65536,
                        flags=sg.F_NO_HOST_SLOTS | sg.F_FORCE_GENERIC) as c:
            forced = run_device(torch, c, pa, rna)
        assert np.all(forced.seq_order[lens_ > 0] == 1)
        assert_same_events(forced, res)


# ---- arbitrary floats --------------------------------------------------------------------------------------------------
def normalised(rng, n, rna):
    rd = synth.make_read(int(rng.integers(1 << 30)), n, seed=77, p_change=0.025 if rna else 0.1)
    x = rd[0].astype(np.float32) * np.float32(0.17) + np.float32(rng.normal(0, 0.01))
    med = np.median(x)
    mad = max(float(np.median(np.abs(x - med))), 1e-3)
    return ((x - med) / np.float32(mad)).astype(np.float32)


def arbitrary_signals(rna):
    rng = np.random.default_rng(900 + rna)
    w2 = 14 if rna else 6
    out = [normalised(rng, int(n), rna) for n in rng.integers(200, 30000, 24)]
    sub = (rng.integers(-40, 40, 5000) * np.float32(2.0 ** -149)).astype(np.float32)
    sub[::4] = 0.0
    out += [sub, np.zeros(3000, np.float32), -np.zeros(700, np.float32)]
    out += [np.full(n, v, np.float32) for n, v in ((4000, 87.5), (999, -3.25e-3), (5000, 1e30))]
    out += [normalised(rng, n, rna) if n else np.zeros(0, np.float32) for n in (0, 1, 2 * w2 - 1, 199, 2 * w2, 200)]
    out += [normalised(rng, 2_000_000, rna), (normalised(rng, 2_000_000, rna) * 1e-20).astype(np.float32)]
    big = normalised(rng, 50000, rna)
    big[1000:1010] = 3e38            # finite, but its window sums overflow float and its squares overflow
    out.append(big)
    for bad in (np.nan, np.inf, -np.inf):
        x = normalised(rng, 20000, rna)
        x[rng.integers(0, 20000, 3)] = bad
        out.append(x)
    x = normalised(rng, 9000, rna)
    x[4500] = np.nan
    x[7000] = np.inf
    out.append(x)
    order = rng.permutation(len(out))
    return [out[i] for i in order]


@pytest.mark.parametrize("rna", [0, 1])
def test_arbitrary_floats(torch, ctx, orc, rna):
    signals = arbitrary_signals(rna)
    res = ctx.run_pa(signals, rna=rna)
    check_oracle(orc, res, signals, rna)
    for r, s in enumerate(signals):
        assert res.seq_order[r] == (0 if len(s) == 0 or witness(s) else 1), f"read {r} ({len(s)} samples): routing"
    assert_same_events(run_device(torch, ctx, signals, rna), res)


def test_huge_reads_alone(torch, orc, sm):
    """three 2,000,000-sample reads alone in a batch: 489 tiles each, shared by many CTAs"""
    reads = [synth.make_read(k, 2_000_000, seed=31) for k in range(3)]
    with sg.Context(device=0, max_samples=1 << 24, max_reads=16) as c:
        pa = c.run(reads, rna=0, want=sg.WANT_PA).pa
        for rna in (0, 1):
            res = c.run_pa(pa, rna=rna)
            assert np.all(res.seq_order == 0)
            check_oracle(orc, res, pa, rna)
            assert_same_events(res, c.run(reads, rna=rna, want=sg.WANT_EVENTS))


# ---- routing ------------------------------------------------------------------------------------------------------------
def test_routing(torch, ctx, orc):
    rng = np.random.default_rng(515)
    good = ctx.run([synth.make_read(k, int(n), seed=515) for k, n in enumerate(rng.integers(100, 40000, 60))],
                   rna=0, want=sg.WANT_PA).pa
    res = ctx.run_pa(good, rna=0)
    assert np.all(res.seq_order == 0)
    check_oracle(orc, res, good, 0)
    mixed, failing = [], []
    for k, s in enumerate(good):
        if k % 3 == 1:
            x = s.copy()
            x[::50] *= np.float32(1e6)       # wide dynamic range: the sums round
            s = x
        mixed.append(s)
        failing.append(not witness(s))
    assert sum(failing) >= 15
    res = ctx.run_pa(mixed, rna=0)
    assert np.array_equal(res.seq_order.astype(bool), np.array(failing))
    check_oracle(orc, res, mixed, 0)
    with sg.Context(device=0, max_samples=1 << 24, max_reads=8192, flags=sg.F_FORCE_GENERIC) as c:
        forced = c.run_pa(mixed, rna=0)
    assert np.all(forced.seq_order == 1)
    assert_same_events(forced, res)


# ---- errors, capacity, scratch, streams ----------------------------------------------------------------------------------
def test_mixed_slots_and_want_bits(torch, ctx):
    lib, h = ctx._lib, ctx._h
    raw = np.arange(100, dtype=np.int16)
    pa = np.linspace(50, 90, 100).astype(np.float32)
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    assert lib.sgpu_slot_add_read(h, 0, raw.ctypes.data, 100, 8192.0, 0.0, 1000.0) == 0
    assert lib.sgpu_slot_add_read_pa(h, 0, pa.ctypes.data, 100) == E_STATE
    assert lib.sgpu_slot_reset(h, 0, 0) == 0
    assert lib.sgpu_slot_add_read_pa(h, 0, pa.ctypes.data, 100) == 0
    assert lib.sgpu_slot_add_read(h, 0, raw.ctypes.data, 100, 8192.0, 0.0, 1000.0) == E_STATE
    stream = Oracle().svbzd_encode(raw)
    assert lib.sgpu_slot_add_read_svbzd(h, 0, stream.ctypes.data, stream.shape[0], 8192.0, 0.0, 1000.0) == E_STATE
    for want in (sg.WANT_PA, sg.WANT_STAT, sg.WANT_EVENTS | sg.WANT_PA, sg.WANT_ENT, sg.WANT_JNN, sg.WANT_PREFIX, 0):
        assert lib.sgpu_submit(h, 0, want) == E_INVAL, want
    ctx.submit(0, sg.WANT_EVENTS)
    assert ctx.wait(0, sg.WANT_EVENTS).events(0).n >= 1
    with pytest.raises(sg.SgpuError) as e:
        ctx.run_device_pa(0, 0, 0, 0, 0, 0, sg.WANT_EVENTS | sg.WANT_STAT)
    assert e.value.code == E_INVAL


def test_capacity_boundaries(orc):
    """a pA slot holds max_samples / 2 floats, every read padded to 8"""
    with sg.Context(device=0, max_samples=4096, max_reads=8) as c:
        lib, h = c._lib, c._h
        x = np.random.default_rng(1).normal(100, 10, 2049).astype(np.float32)
        assert lib.sgpu_slot_reset(h, 0, 0) == 0
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 2049) == sg._lib.E_TOOBIG
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 2048) == 0
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 1) == sg._lib.E_FULL
        assert lib.sgpu_slot_reset(h, 0, 0) == 0
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 1017) == 0     # 1,024 with its padding
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 1025) == sg._lib.E_FULL
        assert lib.sgpu_slot_add_read_pa(h, 0, x.ctypes.data, 1024) == 1
        res = c.run_pa([x[:1017], x[:1024]], rna=0)
        check_oracle(orc, res, [x[:1017], x[:1024]], 0)
        empty = c.run_pa([], rna=0)
        assert empty.n_reads == 0 and np.array_equal(empty.ev_off, np.zeros(1, np.uint64))
        zeros = c.run_pa([np.zeros(0, np.float32)] * 3, rna=1)
        assert np.array_equal(zeros.ev_off, np.zeros(4, np.uint64)) and np.all(zeros.seq_order == 0)


def test_scratch_grows(torch):
    """a context of 96 Mi samples starts with 12 Mi samples of sequential-order scratch; a 40 M-sample pA batch grows it
    and is exact, and the int16 batches before and after (whose own fallback reads fit in an eighth) agree"""
    reads = [synth.make_read(k, 2_000_000, seed=919) for k in range(20)]
    with sg.Context(device=0, max_samples=96 << 20, max_reads=64, flags=sg.F_NO_HOST_SLOTS) as c:
        flat, off, lens = layout([rd[0] for rd in reads])
        dev = torch.device("cuda:0")
        raw16 = np.zeros(flat.shape[0], np.int16)
        for r, rd in enumerate(reads):
            raw16[off[r]:off[r] + lens[r]] = rd[0]
        d_s, d_off = torch.from_numpy(raw16).to(dev), torch.from_numpy(off).to(dev)
        d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
        d_o = torch.tensor([np.float32(rd[2]) for rd in reads], dtype=torch.float32, device=dev)
        d_u = torch.tensor([np.float32(np.float32(rd[3]) / np.float32(rd[1])) for rd in reads], dtype=torch.float32,
                           device=dev)
        span = int(off[-1])
        premise("span (samples) over the initial scratch", span, (96 << 20) // 8)

        def int16_run():
            torch.cuda.synchronize()
            d = c.run_device(d_s.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_o.data_ptr(), d_u.data_ptr(),
                             len(reads), span, 0, sg.WANT_EVENTS | sg.WANT_PA, 0)
            torch.cuda.synchronize()
            ne = c.counters()["n_events"]
            return (c.d2h(d.ev_off, np.uint64, len(reads) + 1), c.d2h(d.ev_start, np.uint32, ne),
                    bits(c.d2h(d.ev_mean, np.float32, ne)), bits(c.d2h(d.ev_stdv, np.float32, ne)),
                    c.d2h(d.pa, np.float32, span))

        before = int16_run()
        pa = [before[4][off[r]:off[r] + lens[r]].copy() for r in range(len(reads))]
        res = run_device(torch, c, pa, 0)
        assert np.all(res.seq_order == 0)
        assert np.array_equal(res.ev_off, before[0]) and np.array_equal(res.ev_start, before[1])
        assert np.array_equal(bits(res.ev_mean), before[2]) and np.array_equal(bits(res.ev_stdv), before[3])
        after = int16_run()
        for a, b in zip(before, after):
            assert np.array_equal(bits(a), bits(b))
        assert_same_events(run_device(torch, c, pa, 0), res)


def test_device_entry_on_a_side_stream(torch, ctx, orc):
    rng = np.random.default_rng(77)
    signals = [normalised(rng, int(n), 0) for n in rng.integers(100, 20000, 40)]
    s = torch.cuda.Stream()
    res = run_device(torch, ctx, signals, 0, stream=s)
    check_oracle(orc, res, signals, 0)

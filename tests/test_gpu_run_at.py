"""GPU tests of reads at any sample offset (sgpu_run_device_at / sgpu_run_device_pa_at, Context.run_device_at /
run_device_pa_at, stage.cu).

Every output of a run on reads at any offset must equal, bit for bit, what sgpu_run_device (sgpu_run_device_pa) returns
for an aligned copy of the same reads that the test builds itself: the staged layout (read_off = stage_off, the last
entry the span), `pa` and the jnn segments taken through stage_off. Covered: every want alone and all together, every
residue of read_off % 8, sample arrays whose base is misaligned by 1..7 elements (tensor slices), packed reads without
gaps, overlapping windows, a window that ends at n_samples, reads of 0, 1, 7, 8, 9 and 200 samples, a 2,000,000-sample
read at an odd offset, a batch large enough that the gather's grid-stride loop comes round more than once, the caller's
detector, jnn and prefix sets, a non-default stream. Trimmed reads are checked against the oracle's getevents on the
sub-array; refused reads (past n_samples, past the span) come back as empty records with the other reads exact."""
import ctypes as C
import os

import numpy as np
import pytest

import _fmt
from _device_out import assert_same, collect
from _oracle import Oracle
from _oracle_pa import getevents_pa
import sigtk_b200 as sg
from sigtk_b200 import _lib as _sl
from sigtk_b200 import synth

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_INVAL, E_TOOBIG = -1, -5
ALL_WANTS = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
STAGE_LAUNCHES = 4  # stage_count, scan, stage_offsets, stage_gather


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 26, max_reads=16384, n_slots=0, flags=sg.F_NO_HOST_SLOTS) as c:
        yield c


@pytest.fixture(autouse=True)
def no_sets(ctx):
    ctx.set_detector(None); ctx.set_jnn(None); ctx.set_prefix(None)
    yield
    ctx.set_detector(None); ctx.set_jnn(None); ctx.set_prefix(None)


def align8(n):
    return (np.asarray(n, np.int64) + 7) // 8 * 8


def calib(reads):
    """offset_f, raw_unit_f as sgpu_slot_add_read forms them (misc.c:17-19,26)"""
    return (np.array([np.float32(rd[2]) for rd in reads], np.float32),
            np.array([np.float32(rd[3]) / np.float32(rd[1]) for rd in reads], np.float32))


def expected_stage(read_off, read_len, n_samples, span):
    """stage_off and the staged lengths the header promises (refused reads staged as empty records); -> (off, len,
    status)"""
    read_off, read_len = np.asarray(read_off, np.uint64), np.asarray(read_len, np.uint64)
    ok = (read_off <= n_samples) & (read_len <= np.uint64(n_samples) - np.minimum(read_off, np.uint64(n_samples)))
    g = np.where(ok, (read_len.astype(np.int64) + 7) // 8, 0)
    goff = np.zeros(len(g) + 1, np.int64)
    goff[1:] = np.cumsum(g)
    fits = 8 * goff[1:] <= span
    off = np.minimum(8 * goff, span)
    ln = np.where(ok & fits, read_len.astype(np.int64), 0)
    status = E_INVAL if not ok.all() else (E_TOOBIG if not fits.all() else 0)
    return off.astype(np.uint64), ln, status


class Run:
    """the result of one run: outputs, stage_off, staged lengths, counters"""

    def __init__(self, out, stage_off, lens, counters):
        self.out, self.stage_off, self.lens, self.counters = out, stage_off, lens, counters


def run_at(torch, ctx, samples, read_off, read_len, reads_calib, span, rna, want, stream=None, n_samples=None):
    """sgpu_run_device_at on the torch int16 tensor `samples` (any slice) with the reads (read_off, read_len)"""
    dev = samples.device
    n = len(read_len)
    d_off = torch.from_numpy(np.asarray(read_off, np.uint64).view(np.int64)).to(dev)
    d_len = torch.from_numpy(np.asarray(read_len, np.uint32).view(np.int32)).to(dev)
    d_o, d_u = (torch.from_numpy(x).to(dev) for x in reads_calib)
    torch.cuda.synchronize()
    st = (stream or torch.cuda.current_stream()).cuda_stream
    d, soff = ctx.run_device_at(samples.data_ptr(), samples.numel() if n_samples is None else n_samples,
                                d_off.data_ptr(), d_len.data_ptr(), d_o.data_ptr(), d_u.data_ptr(), n, span, rna, want,
                                st)
    torch.cuda.synchronize()
    c = ctx.counters()
    stage_off = ctx.d2h(soff, np.uint64, n + 1)
    exp_off, exp_len, exp_status = expected_stage(read_off, read_len, samples.numel() if n_samples is None else n_samples,
                                                  span)
    assert np.array_equal(stage_off, exp_off), "stage_off is not the promised layout"
    assert c["status"] == exp_status, c
    return Run(collect(ctx, d, n, stage_off, exp_len, want, span), stage_off, exp_len, c)


def run_aligned(torch, ctx, reads_raw, run, reads_calib, span, rna, want, stream=None):
    """sgpu_run_device on an aligned copy of the reads in the staged layout of `run` (read_off[n] = span)"""
    n = len(reads_raw)
    flat = np.zeros(max(span, 8), np.int16)
    for r in range(n):
        k = int(run.lens[r])
        flat[int(run.stage_off[r]): int(run.stage_off[r]) + k] = reads_raw[r][:k]
    off = run.stage_off.copy()
    off[n] = span
    dev = torch.device("cuda:0")
    arrs = [torch.from_numpy(x).to(dev) for x in (flat, off.view(np.int64), run.lens.astype(np.int32), *reads_calib)]
    torch.cuda.synchronize()
    st = (stream or torch.cuda.current_stream()).cuda_stream
    d = ctx.run_device(*[a.data_ptr() for a in arrs], n, span, rna, want, st)
    torch.cuda.synchronize()
    c = ctx.counters()
    assert c["status"] == 0
    return collect(ctx, d, n, off, run.lens, want, span), c


def packed(reads, base_shift, torch, gap=None):
    """the reads back to back without padding from element `base_shift` of a tensor (a slice of it: its data_ptr is
    misaligned by base_shift elements); -> (tensor slice, read_off, read_len)"""
    lens = np.array([len(rd[0]) for rd in reads], np.int64)
    off = np.zeros(len(reads), np.int64)
    if len(reads) > 1:
        off[1:] = np.cumsum(lens[:-1])
    total = int(lens.sum())
    flat = np.zeros(base_shift + total + 3, np.int16)
    for r, rd in enumerate(reads):
        flat[base_shift + off[r]: base_shift + off[r] + lens[r]] = rd[0]
    t = torch.from_numpy(flat).to("cuda:0")
    sl = t[base_shift: base_shift + total]
    return sl, off.astype(np.uint64), lens.astype(np.uint32)


def check_against_aligned(torch, ctx, samples, read_off, read_len, reads, rna, want, span=None, stream=None):
    """run at any offset and on the aligned copy, compare every output; -> the Run"""
    host = samples.cpu().numpy()
    raws = [host[int(o): int(o) + int(n)] for o, n in zip(read_off, read_len)]
    if span is None:
        span = int(align8(read_len).sum()) + 64
    cal = calib(reads)
    run = run_at(torch, ctx, samples, read_off, read_len, cal, span, rna, want, stream)
    ref, c = run_aligned(torch, ctx, raws, run, cal, span, rna, want, stream)
    assert_same(run.out, ref, f"want {want} rna {rna}")
    assert run.counters["n_kernel_launches"] == c["n_kernel_launches"] + (STAGE_LAUNCHES if len(reads) else 0)
    return run


def make_read(k, n, seed):
    """synth.make_read, also for n = 0"""
    rd = synth.make_read(k, max(n, 1), seed=seed)
    return (rd[0][:n].copy(),) + tuple(rd[1:])


def mixed_reads(n, rna, seed):
    """reads of 0, 1, 7, 8, 9 and 200 samples among lengths of a few hundred to 30,000"""
    rng = np.random.default_rng(seed)
    lens = list(rng.integers(100, 30000, n))
    lens[1:7] = [0, 1, 7, 8, 9, 200]
    if rna:
        return synth.make_reads(n, mean=20000.0, seed=seed, rna=True)[:n - 6] + \
            [make_read(1000 + k, int(m), seed) for k, m in enumerate([0, 1, 7, 8, 9, 200])]
    return [make_read(k, int(m), seed) for k, m in enumerate(lens)]


# ---- equality with the aligned path -------------------------------------------------------------------------------
@pytest.mark.parametrize("rna", [0, 1])
@pytest.mark.parametrize("want", [sg.WANT_EVENTS, sg.WANT_PA, sg.WANT_STAT, sg.WANT_ENT, sg.WANT_JNN, sg.WANT_PREFIX,
                                  ALL_WANTS])
def test_every_want_packed(torch, ctx, want, rna):
    reads = mixed_reads(120, rna, 700 + rna)
    samples, off, lens = packed(reads, 3, torch)
    assert set((off % 8).tolist()) == set(range(8)), "every residue of read_off % 8"
    check_against_aligned(torch, ctx, samples, off, lens, reads, rna, want)


@pytest.mark.parametrize("shift", range(1, 8))
def test_misaligned_base(torch, ctx, shift):
    """a tensor slice whose data_ptr is 2 * shift bytes past a 16-byte boundary"""
    reads = mixed_reads(40, 0, 810 + shift)
    samples, off, lens = packed(reads, shift, torch)
    assert samples.data_ptr() % 16 == 2 * shift
    check_against_aligned(torch, ctx, samples, off, lens, reads, 0, ALL_WANTS)


def test_overlapping_windows(torch, ctx):
    """windows of one read that overlap, nest and repeat, one ending exactly at n_samples"""
    rd = synth.make_read(0, 100_003, seed=91)
    t = torch.from_numpy(rd[0].copy()).to("cuda:0")
    n = t.numel()
    wins = [(0, n), (5, 1000), (6, 1000), (13, 99_000), (n - 777, 777), (n - 1, 1), (n, 0), (50_000, 50_003),
            (0, 0), (3, 200), (3, 200), (40_001, 9)]
    off = np.array([w[0] for w in wins], np.uint64)
    lens = np.array([w[1] for w in wins], np.uint32)
    reads = [rd] * len(wins)
    check_against_aligned(torch, ctx, t, off, lens, reads, 0, ALL_WANTS)


def test_two_million_samples_at_an_odd_offset(torch, ctx):
    long = synth.make_read(0, 2_000_000, seed=92)
    reads = [synth.make_read(1, 13, seed=92), long, synth.make_read(2, 5, seed=92)]
    samples, off, lens = packed(reads, 1, torch)
    assert off[1] % 2 == 1
    check_against_aligned(torch, ctx, samples, off, lens, reads, 0, ALL_WANTS)


def test_grid_stride_loops_come_round(torch, ctx):
    """12,000 reads packed from an odd base: the gather's grid (sm x 16 CTAs x 8,192 samples) takes more than one step"""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(93)
    lens = rng.integers(0, 8000, 12000)
    reads = [make_read(k, int(m), 93) for k, m in enumerate(lens)]
    samples, off, lens = packed(reads, 5, torch)
    span = int(align8(lens).sum())
    assert span > 2 * sm * 16 * 8192
    check_against_aligned(torch, ctx, samples, off, lens, reads, 0, ALL_WANTS, span=span)


def test_with_the_callers_sets(torch, ctx):
    """a detector, a jnn and a prefix set in force apply as in sgpu_run_device"""
    reads = mixed_reads(60, 1, 94)
    samples, off, lens = packed(reads, 7, torch)
    ctx.set_detector(sg.Detector(4, 9, 2.0, 8.0, 0.5))
    ctx.set_jnn(sg.Jnn(188, 0.25, 4, 60, 50, 0.7))
    ctx.set_prefix(sg.Prefix(sg.Adaptor(1337, 0.6, 1200, 800, 150000), sg.Polya(200, 1.0, 25, 150, 40)))
    check_against_aligned(torch, ctx, samples, off, lens, reads, 1, ALL_WANTS)


def test_non_default_stream_and_forced_generic(torch):
    """a run on a stream of the caller's, in a context that sends every read through the sequential-order kernels"""
    reads = mixed_reads(50, 0, 95)
    with sg.Context(device=0, max_samples=1 << 22, max_reads=256, n_slots=0,
                    flags=sg.F_NO_HOST_SLOTS | sg.F_FORCE_GENERIC | sg.F_STAGE_TIMERS) as c:
        s = torch.cuda.Stream()
        samples, off, lens = packed(reads, 3, torch)
        with torch.cuda.stream(s):
            check_against_aligned(torch, c, samples, off, lens, reads, 0, ALL_WANTS, stream=s)
            run_at(torch, c, samples, off, lens, calib(reads), int(align8(lens).sum()), 0, sg.WANT_EVENTS, stream=s)
        names = [st[0] for st in c.stage_times()]
        assert names[0] == "stage_reads" and c.stage_times()[0][2] == STAGE_LAUNCHES


def test_pa_reads_at_any_offset(torch, ctx, orc):
    """pA floats packed from a base misaligned by 1..3 floats, and overlapping windows, against sgpu_run_device_pa on
    an aligned copy; the events equal the oracle's getevents(n, pa, rna)"""
    for rna, shift in ((0, 1), (1, 2), (0, 3)):
        reads = mixed_reads(80, rna, 960 + shift)
        sigs = [orc.pa(*rd) for rd in reads]
        lens = np.array([len(s) for s in sigs], np.int64)
        off = np.zeros(len(sigs), np.int64)
        off[1:] = np.cumsum(lens[:-1])
        flat = np.zeros(shift + int(lens.sum()), np.float32)
        for r, s in enumerate(sigs):
            flat[shift + off[r]: shift + off[r] + lens[r]] = s
        sigs.append(flat[shift + 11: shift + 4000].copy())  # a window across the first reads
        off, lens = np.append(off, 11), np.append(lens, 3989)
        t = torch.from_numpy(flat).to("cuda:0")[shift:]
        span = int(align8(lens).sum())
        d_off = torch.from_numpy(off).to("cuda:0")
        d_len = torch.from_numpy(lens.astype(np.int32)).to("cuda:0")
        torch.cuda.synchronize()
        d, soff = ctx.run_device_pa_at(t.data_ptr(), t.numel(), d_off.data_ptr(), d_len.data_ptr(), len(sigs), span,
                                       rna, sg.WANT_EVENTS, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert ctx.counters()["status"] == 0
        n = len(sigs)
        stage_off = ctx.d2h(soff, np.uint64, n + 1)
        exp_off, exp_len, _ = expected_stage(off, lens, t.numel(), span)
        assert np.array_equal(stage_off, exp_off)
        got = collect(ctx, d, n, stage_off, exp_len, sg.WANT_EVENTS, span)
        # the aligned copy
        a = np.zeros(span, np.float32)
        for r, s in enumerate(sigs):
            a[int(stage_off[r]): int(stage_off[r]) + len(s)] = s
        aoff = stage_off.copy()
        aoff[n] = span
        d_a, d_ao = torch.from_numpy(a).to("cuda:0"), torch.from_numpy(aoff.view(np.int64)).to("cuda:0")
        torch.cuda.synchronize()
        d2 = ctx.run_device_pa(d_a.data_ptr(), d_ao.data_ptr(), d_len.data_ptr(), n, span, rna)
        torch.cuda.synchronize()
        ref = collect(ctx, d2, n, aoff, exp_len, sg.WANT_EVENTS, span)
        assert_same(got, ref, f"pA rna {rna} shift {shift}")
        for r in (0, 1, 5, n - 1):
            res = sg.BatchResult(n_reads=n, read_len=lens.astype(np.uint32), ev_off=got["ev_off"],
                                 ev_start=got["ev_start"], ev_mean=got["ev_mean"].view(np.float32),
                                 ev_stdv=got["ev_stdv"].view(np.float32))
            ev = res.events(r)
            if lens[r] == 0:
                assert ev.n == 0
                continue
            st, ln, mn, sd = getevents_pa(orc, sigs[r], rna)
            assert np.array_equal(ev.start, st) and np.array_equal(ev.mean.view(np.uint32), mn.view(np.uint32))
            assert np.array_equal(ev.stdv.view(np.uint32), sd.view(np.uint32))


# ---- against the reference's arithmetic: trimmed reads ----------------------------------------------------------------
@pytest.mark.parametrize("npz,rna", [("synth_rna.npz", 1), ("sp1_dna.npz", 0)])
def test_trimmed_reads_against_the_oracle(torch, ctx, orc, npz, rna):
    """prefix (RNA: the adaptor's end, then the poly-A's) or jnn (DNA: the first stall's end) found by a
    device-resident run, then the events of [start, n) of every read as getevents on the sub-array, int16 and pA"""
    reads = [rd for _, rd in _fmt.load_npz(os.path.join(G, npz))]
    samples, off, lens = packed(reads, 0, torch)
    span = int(align8(lens).sum())
    want = sg.WANT_PREFIX if rna else sg.WANT_JNN
    run = run_at(torch, ctx, samples, off, lens, calib(reads), span, rna, want)
    n = len(reads)
    if rna:
        pos = run.out["prefix_pos"].reshape(n, 4).astype(np.int64)
        start = np.where(pos[:, 1] > 0, pos[:, 1] + np.where(pos[:, 3] > 0, pos[:, 3], 0), 0)
    else:
        start = np.array([int(s[0][1]) if len(s) else 0 for s in run.out["jnn"]], np.int64)
    start = np.clip(start, 0, lens.astype(np.int64))
    assert (start > 0).any(), "premise: some reads are trimmed"
    # read_off' = read_off + start, read_len' = n - start, computed on the device
    d_start = torch.from_numpy(start).to("cuda:0")
    t_off = torch.from_numpy(off.view(np.int64)).to("cuda:0") + d_start
    t_len = (torch.from_numpy(lens.astype(np.int64)).to("cuda:0") - d_start).to(torch.int32)
    new_off, new_len = t_off.cpu().numpy().view(np.uint64), t_len.cpu().numpy().view(np.uint32)
    trimmed = run_at(torch, ctx, samples, new_off, new_len, calib(reads), span, rna, sg.WANT_EVENTS)
    ev_off = trimmed.out["ev_off"]
    pa_all = []
    for r, rd in enumerate(reads):
        sub = rd[0][start[r]:]
        a, b = int(ev_off[r]), int(ev_off[r + 1])
        if len(sub) == 0:
            assert a == b
            pa_all.append(np.zeros(0, np.float32))
            continue
        st, ln, mn, sd = orc.events(sub, rd[1], rd[2], rd[3], rna=rna)
        assert np.array_equal(trimmed.out["ev_start"][a:b], st.astype(np.uint32)), f"read {r}: event starts"
        assert np.array_equal(trimmed.out["ev_mean"][a:b], mn.view(np.uint32)), f"read {r}: means"
        assert np.array_equal(trimmed.out["ev_stdv"][a:b], sd.view(np.uint32)), f"read {r}: stdv"
        pa_all.append(orc.pa(*rd))
    # the same on pA sub-arrays
    flat = np.concatenate(pa_all) if pa_all else np.zeros(0, np.float32)
    poff = np.zeros(n, np.int64)
    poff[1:] = np.cumsum([len(p) for p in pa_all])[:-1]
    plen = np.array([len(p) for p in pa_all], np.int64)
    t = torch.from_numpy(flat).to("cuda:0")
    d_off = torch.from_numpy(poff + np.minimum(start, plen)).to("cuda:0")
    d_len = torch.from_numpy((plen - np.minimum(start, plen)).astype(np.int32)).to("cuda:0")
    torch.cuda.synchronize()
    d, soff = ctx.run_device_pa_at(t.data_ptr(), t.numel(), d_off.data_ptr(), d_len.data_ptr(), n, span, rna)
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0
    got = collect(ctx, d, n, ctx.d2h(soff, np.uint64, n + 1), plen - np.minimum(start, plen), sg.WANT_EVENTS, span)
    for r in range(n):
        if len(pa_all[r]) <= start[r]:
            continue
        st, ln, mn, sd = getevents_pa(orc, pa_all[r][start[r]:], rna)
        a, b = int(got["ev_off"][r]), int(got["ev_off"][r + 1])
        assert np.array_equal(got["ev_start"][a:b], st.astype(np.uint32)), f"pA read {r}: event starts"
        assert np.array_equal(got["ev_mean"][a:b], mn.view(np.uint32)), f"pA read {r}: means"


# ---- refusals and status -----------------------------------------------------------------------------------------------
def test_host_refusals(torch, ctx):
    reads = mixed_reads(10, 0, 97)
    samples, off, lens = packed(reads, 1, torch)
    dev = torch.device("cuda:0")
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    d_len = torch.from_numpy(lens.view(np.int32)).to(dev)
    d_o, d_u = (torch.from_numpy(x).to(dev) for x in calib(reads))
    span = int(align8(lens).sum())
    n = len(reads)
    lib, h = ctx._lib, ctx._h

    def at(samples_ptr=samples.data_ptr(), n_samples=samples.numel(), o=d_off.data_ptr(), ln=d_len.data_ptr(),
           of=d_o.data_ptr(), u=d_u.data_ptr(), nr=n, sp=span, want=ALL_WANTS):
        db = _sl.DevReads(samples_ptr, n_samples, o, ln, of, u, nr, 0, sp)
        res, so = _sl.Result(), C.c_void_p()
        return lib.sgpu_run_device_at(h, C.byref(db), want, None, C.byref(res), C.byref(so))

    def pa_at(pa_ptr, nr=n, sp=span, want=sg.WANT_EVENTS):
        db = _sl.DevPaReads(pa_ptr, samples.numel(), d_off.data_ptr(), d_len.data_ptr(), nr, 0, sp)
        res, so = _sl.Result(), C.c_void_p()
        return lib.sgpu_run_device_pa_at(h, C.byref(db), want, None, C.byref(res), C.byref(so))

    assert at(nr=ctx.max_reads + 1) == E_INVAL
    assert at(sp=ctx.max_samples + 8) == E_INVAL
    assert at(sp=span + 4) == E_INVAL
    assert at(o=0) == E_INVAL and at(ln=0) == E_INVAL and at(samples_ptr=0) == E_INVAL
    assert at(of=0) == E_INVAL and at(u=0, want=sg.WANT_STAT) == E_INVAL and at(u=0, want=sg.WANT_PREFIX) == E_INVAL
    assert at(want=sg.WANT_EVENTS | sg.WANT_SVBZD) == E_INVAL and at(want=0) == E_INVAL
    assert at(samples_ptr=samples.data_ptr() + 1) == E_INVAL  # not 2-byte aligned
    f = torch.zeros(64, dtype=torch.float32, device=dev)
    assert pa_at(f.data_ptr(), want=sg.WANT_PA) == E_INVAL and pa_at(f.data_ptr() + 2) == E_INVAL
    assert pa_at(f.data_ptr(), sp=span + 4) == E_INVAL
    # (offset_f / raw_unit_f are not read by ENT and JNN)
    torch.cuda.synchronize()
    assert at(of=0, u=0, want=sg.WANT_ENT | sg.WANT_JNN) == 0
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0


@pytest.mark.parametrize("case", ["past_n_samples", "past_span", "both"])
def test_device_refusals(torch, ctx, case):
    """refused reads come back as empty records, the others exact; the next valid run is exact again"""
    reads = mixed_reads(60, 0, 98)
    samples, off, lens = packed(reads, 3, torch)
    span = int(align8(lens).sum())
    off, lens = off.copy(), lens.copy()
    if case in ("past_n_samples", "both"):
        lens[10] = samples.numel() - int(off[10]) + 1      # one sample past the end
        off[20] = samples.numel() + 5                        # starts past the end
        off[30], lens[30] = 2**64 - 4, 8                     # wraps around
    if case in ("past_span", "both"):                        # reads 45.. no longer fit
        span = int(align8(expected_stage(off, lens, samples.numel(), 1 << 62)[1][:45]).sum()) + 8
    host = samples.cpu().numpy()
    raws = [host[int(o): int(o) + int(n)] if int(o) + int(n) <= len(host) else np.zeros(0, np.int16)
            for o, n in zip(off, lens)]
    cal = calib(reads)
    run = run_at(torch, ctx, samples, off, lens, cal, span, 0, ALL_WANTS)
    assert run.counters["status"] == (E_TOOBIG if case == "past_span" else E_INVAL)
    refused = np.nonzero(run.lens != lens.astype(np.int64))[0]
    assert len(refused) >= 3
    ev_off = run.out["ev_off"]
    assert all(ev_off[r] == ev_off[r + 1] for r in refused)
    ref, _ = run_aligned(torch, ctx, raws, run, cal, span, 0, ALL_WANTS)
    assert_same(run.out, ref, case)
    good_off, good_len = packed(reads, 3, torch)[1:]
    check_against_aligned(torch, ctx, samples, good_off, good_len, reads, 0, ALL_WANTS)


def test_no_reads(torch, ctx):
    t = torch.zeros(16, dtype=torch.int16, device="cuda:0")
    d, soff = ctx.run_device_at(t.data_ptr(), 16, 0, 0, 0, 0, 0, 0, 0, sg.WANT_EVENTS)
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0
    assert ctx.d2h(soff, np.uint64, 1)[0] == 0 and ctx.d2h(d.ev_off, np.uint64, 1)[0] == 0

"""The statistics of pA records (SGPU_WANT_STAT on pA slots, sgpu_run_device_pa, sgpu_run_device_pa_at): meanf, stdvf,
medianf of the caller's floats in columns 1, 3, 5 of `stat`, a NaN in columns 0, 2, 4.

- Round trip: the pA of an int16 run fed back in gives that run's columns 1, 3, 5 bit for bit.
- Arbitrary floats (normalised signal, signed running sums aimed at the signed summaries of float_order.cuh, NaN, Inf,
  subnormals, -0) against the plain sequential reference of tests/_stat_ref.py: mean and stdv bit for bit (NaN where
  the reference's are NaN), the median bit for bit except a zero, which is compared by value, and NaN for a read that
  holds a NaN.
- Both roles of the moments kernel (PARAM_STAT_CTA_MIN 0: a CTA per read; 2^31: a warp per read) and the default.
- Which wants a pA record accepts (STAT only in a context opened with SGPU_F_PA_STAT), and that a STAT-only run
  launches no event kernel."""
import ctypes as C
import os

import numpy as np
import pytest

import _fmt
import _stat_ref as R
import sigtk_b200 as sg
from sigtk_b200 import _lib as _sl, synth
from test_gpu_pa_input import arbitrary_signals, assert_same_events, layout

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_INVAL, E_STATE = -1, -6
CTA_MIN_DEFAULT = 131072
ROLES = [0, CTA_MIN_DEFAULT, 1 << 31]
F = np.float32


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 25, max_reads=16384, flags=sg.F_STAGE_TIMERS | sg.F_PA_STAT) as c:
        yield c


@pytest.fixture(autouse=True)
def defaults(ctx):
    yield
    ctx.set_param(_sl.PARAM_STAT_CTA_MIN, CTA_MIN_DEFAULT)


def bits(a):
    return np.asarray(a, F).view(np.uint32)


def seq_sum(x):
    """float acc = 0; for (...) acc = acc + x[i]: from +0, as stat.h's loops (a read of -0.0 sums to +0)"""
    with np.errstate(all="ignore"):
        return np.add.accumulate(np.concatenate([[F(0.0)], np.asarray(x, F)]), dtype=F)[-1]


def ref3(x):
    """meanf, stdvf, medianf of one record: sequential float32 loops, the element of rank n // 2 (NaN when the record
    holds a NaN); an empty record: 0/0, 0/0, 0"""
    x = np.asarray(x, F)
    if len(x) == 0:
        return np.array([np.nan, np.nan, 0.0], F)
    n = F(len(x))
    with np.errstate(all="ignore"):
        mean = seq_sum(x) / n
        stdv = np.sqrt(seq_sum(R.squares(x, mean)) / n)
    med = F(np.nan) if np.isnan(x).any() else R.rank_half(x)
    return np.array([mean, stdv, med], F)


def stat_mismatch(row, want):
    """'' when a stat row of a pA record matches ref3's numbers, else what differs"""
    row = np.asarray(row, F)
    if not np.all(np.isnan(row[[0, 2, 4]])):
        return "raw columns not NaN"
    got = row[[1, 3, 5]]
    if not R.same_stat(got[:2], want[:2]):
        return f"mean / stdv {got[:2]} != {want[:2]}"
    if want[2] == 0 and got[2] == 0:
        return ""                                   # -0 and +0: no sort pins which zero is the median
    if not R.same_stat(got[2:], want[2:]):
        return f"median {got[2]!r} != {want[2]!r}"
    return ""


def check_ref(stat, signals, what):
    bad = [(r, len(signals[r]), m) for r in range(len(signals)) if (m := stat_mismatch(stat[r], ref3(signals[r])))]
    assert not bad, f"{what}: {len(bad)} of {len(signals)} reads differ (read, length, what): {bad[:6]}"


def device_run(torch, ctx, signals, want):
    """sgpu_run_device_pa on device copies of `signals` -> (stat [n][6] or None, device result, layout)"""
    flat, off, lens = layout(signals)
    dev = torch.device("cuda:0")
    d_pa, d_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    torch.cuda.synchronize()
    d = ctx.run_device_pa(d_pa.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), len(signals), int(off[-1]), 0, want,
                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0
    n = len(signals)
    stat = ctx.d2h(d.stat, F, 6 * n).reshape(n, 6) if want & sg.WANT_STAT else None
    return stat, d, (off, lens)


def device_stat(torch, ctx, signals):
    return device_run(torch, ctx, signals, sg.WANT_STAT)[0]


def device_stat_at(torch, ctx, flat, starts, lens):
    """sgpu_run_device_pa_at on windows flat[starts[r] .. + lens[r]) of one packed array"""
    dev = torch.device("cuda:0")
    d_pa = torch.from_numpy(np.asarray(flat, F)).to(dev)
    d_off = torch.from_numpy(np.asarray(starts, np.int64)).to(dev)
    d_len = torch.from_numpy(np.asarray(lens, np.int32)).to(dev)
    span = int(((np.asarray(lens, np.int64) + 7) // 8 * 8).sum()) or 8
    torch.cuda.synchronize()
    d, _ = ctx.run_device_pa_at(d_pa.data_ptr(), len(flat), d_off.data_ptr(), d_len.data_ptr(), len(lens), span, 0,
                                sg.WANT_STAT, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0
    return ctx.d2h(d.stat, F, 6 * len(lens)).reshape(len(lens), 6)


def all_paths(torch, ctx, signals):
    """{path: stat} for the host slot and sgpu_run_device_pa"""
    return {"host": ctx.run_pa(signals, want=sg.WANT_STAT).stat, "device": device_stat(torch, ctx, signals)}


# ---- round trip: the int16 route's pA fed back in -----------------------------------------------------------------------
def round_trip_batches():
    rng = np.random.default_rng(2024)
    golden = {name: [rd for _, rd in _fmt.load_npz(os.path.join(G, name))] for name in ("sp1_dna.npz", "synth_rna.npz")}
    synthetic = [synth.make_read(k, int(n), seed=2024) for k, n in
                 enumerate([2_000_000, 2_000_000, 1, 7, 31, 33, 500, 1023, 1025, 8191, 131072, 131073] +
                           list(rng.integers(100, 60000, 40)))]
    synthetic.insert(3, (np.zeros(0, np.int16), 8192.0, 4.0, 1400.0))                   # an empty record
    return {**golden, "synthetic": synthetic}


@pytest.mark.parametrize("batch", ["sp1_dna.npz", "synth_rna.npz", "synthetic"])
def test_round_trip(torch, ctx, batch):
    reads = round_trip_batches()[batch]
    for cta_min in ROLES:
        ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
        raw = ctx.run(reads, rna=0, want=sg.WANT_PA | sg.WANT_STAT)
        pa = [p.copy() for p in raw.pa]
        want = raw.stat[:, [1, 3, 5]]
        got = all_paths(torch, ctx, pa)
        # the same records at odd offsets of one packed array, and windows that overlap them
        flat = np.concatenate([np.zeros(3, F)] + pa + [np.zeros(5, F)])
        starts = 3 + np.concatenate([[0], np.cumsum([len(p) for p in pa])[:-1]]).astype(np.int64)
        lens = np.array([len(p) for p in pa], np.int64)
        n_win = min(len(pa), 20)
        w_start = starts[:n_win] + lens[:n_win] // 2
        w_len = np.minimum(lens[:n_win] + 100, len(flat) - w_start)
        at = device_stat_at(torch, ctx, flat, np.concatenate([starts, w_start]), np.concatenate([lens, w_len]))
        got["at"] = at[:len(pa)]
        for path, stat in got.items():
            assert np.all(np.isnan(stat[:, [0, 2, 4]])), (batch, cta_min, path)
            bad = np.nonzero(~np.all(bits(stat[:, [1, 3, 5]]) == bits(want), axis=1))[0]
            assert not len(bad), (batch, cta_min, path, bad[:8], stat[bad[:2]], raw.stat[bad[:2]])
        windows = [flat[int(s):int(s) + int(n)] for s, n in zip(w_start, w_len)]
        check_ref(at[len(pa):], windows, f"{batch} overlapping windows, cta_min {cta_min}")


# ---- arbitrary floats ----------------------------------------------------------------------------------------------------
def signed_signals():
    """reads aimed at the signed summaries: sums of either sign, crossing zero and binade edges, ties"""
    rng = np.random.default_rng(77)
    out = []
    out += [-np.abs(rng.normal(100, 10, n)).astype(F) for n in (700, 5000, 300_000)]           # all negative
    out += [rng.normal(0, 1, n).astype(F) for n in (3000, 200_000)]                             # a random walk around 0
    out += [rng.normal(-0.02, 1, 400_000).astype(F)]                                            # drifting down
    # running sums that return to exactly 0 at tile (32) and superblock (1024) boundaries, and cross it between them
    for period, shift in ((32, 0), (1024, 0), (64, 7), (2048, 511), (8192, 0)):
        base = np.where((np.arange(period) < period // 2), F(0.75), F(-0.75))
        x = np.tile(base, 300_000 // period + 1)[:300_000]
        out.append(np.roll(x, shift).astype(F))
    # a walk around a power of two: sums one ulp under 2^20 and back, steps of half an ulp (ties of both parities)
    for start in (F(2.0 ** 20), F(-(2.0 ** 20)), F(2.0 ** 20 - 0.125)):
        steps = (rng.integers(-3, 4, 200_000) * F(0.0625)).astype(F)
        out.append(np.concatenate([[start], steps]).astype(F))
    # ties at half an ulp far from any binade edge, both parities, either sign of accumulator
    for acc in (F(3.0 * 2 ** 21), F(-3.0 * 2 ** 21)):
        steps = ((rng.integers(0, 2, 100_000) * 2 - 1) * F(0.25)).astype(F)                   # ulp at 3*2^21 is 0.5
        steps[::3] = F(0.75)
        out.append(np.concatenate([[acc], steps]).astype(F))
    # alternating huge and tiny magnitudes
    x = np.empty(50_000, F)
    x[0::2] = (rng.integers(0, 2, 25_000) * 2 - 1) * F(1e20)
    x[1::2] = rng.normal(0, 1e-20, 25_000).astype(F)
    out.append(x)
    x = rng.normal(0, 1, 70_000).astype(F)
    x[::5] = F(-0.0)
    out += [x, np.concatenate([-np.zeros(3000, F), rng.normal(-5, 1, 5000).astype(F)])]          # -0.0 addends
    # normalised signal, both signs, long
    raw = synth.make_read(9, 2_000_000, seed=9)[0].astype(F)
    med = F(np.median(raw))
    mad = F(np.median(np.abs(raw - med)))
    out.append(((raw - med) / mad).astype(F))
    return out


@pytest.mark.parametrize("cta_min", ROLES)
def test_arbitrary_floats(torch, ctx, cta_min):
    ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
    signals = arbitrary_signals(0) + arbitrary_signals(1)[:10] + signed_signals()
    for path, stat in all_paths(torch, ctx, signals).items():
        check_ref(stat, signals, f"{path}, cta_min {cta_min}")


def test_median_edges(torch, ctx):
    rng = np.random.default_rng(5)
    sub = F(2.0 ** -149)
    signals = [np.array([3.5], F), np.array([-2.0], F), np.array([1.0, -1.0], F), np.array([-0.0, 0.0], F),
               np.array([0.0, -0.0, 0.0], F), np.full(4097, 87.25, F), np.full(33, -1e-3, F),
               np.where(rng.random(5000) < 0.5, F(1.5), F(-7.0)).astype(F),
               np.where(rng.random(5001) < 0.5, F(np.inf), F(-np.inf)).astype(F),
               np.array([np.inf, 1.0, -np.inf], F), np.array([np.inf] * 3 + [5.0], F),
               (rng.integers(-40, 40, 10001) * sub).astype(F), (rng.integers(1, 5, 999) * sub).astype(F),
               np.where(rng.random(3001) < 0.5, F(0.0), F(-0.0)).astype(F),
               np.concatenate([np.where(rng.random(2000) < 0.5, F(0.0), F(-0.0)), np.full(1000, 1.0, F),
                               np.full(1000, -1.0, F)]).astype(F),
               np.array([np.nan], F), np.array([1.0, np.nan, 2.0], F),
               (F(1.0) + rng.integers(0, 4096, 2_000_000).astype(F) * F(2.0 ** -23)).astype(F),   # one key prefix
               (-(F(1.0) + rng.integers(0, 256, 1_000_001).astype(F) * F(2.0 ** -23))).astype(F),
               np.zeros(0, F)]
    for cta_min in ROLES:
        ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
        for path, stat in all_paths(torch, ctx, signals).items():
            check_ref(stat, signals, f"{path}, cta_min {cta_min}")
            assert np.isnan(stat[-1, 1]) and np.isnan(stat[-1, 3]) and bits(stat[-1, 5]) == 0   # empty: 0/0, +0


def test_padding_and_stale_slots(torch, ctx):
    """values past read_len never count: NaN / Inf / huge garbage in a device batch's padding, and a host slot whose
    sample buffer held a longer earlier batch"""
    rng = np.random.default_rng(8)
    signals = [rng.normal(0, 1, int(n)).astype(F) for n in (1, 5, 31, 1021, 5003, 140_001)]
    flat, off, lens = layout(signals)
    for r in range(len(signals)):
        flat[off[r] + lens[r]:off[r + 1]] = [np.nan, np.inf, -3e38, 7.0, -np.inf, 1e30, np.nan][:off[r + 1] - off[r] - lens[r]]
    dev = torch.device("cuda:0")
    d_pa, d_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    for cta_min in (0, 1 << 31):
        ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
        torch.cuda.synchronize()
        d = ctx.run_device_pa(d_pa.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), len(signals), int(off[-1]), 0,
                              sg.WANT_STAT, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        check_ref(ctx.d2h(d.stat, F, 6 * len(signals)).reshape(-1, 6), signals, f"device padding, cta_min {cta_min}")
        ctx.run_pa([np.full(200_000, np.nan, F)] * 3, want=sg.WANT_STAT)
        check_ref(ctx.run_pa(signals, want=sg.WANT_STAT).stat, signals, f"stale slot, cta_min {cta_min}")


# ---- wants --------------------------------------------------------------------------------------------------------------
def test_stat_only_launches_no_event_kernel(torch, ctx):
    rng = np.random.default_rng(12)
    signals = [rng.normal(90, 10, int(n)).astype(F) for n in rng.integers(10, 50_000, 50)]
    stat, _, _ = device_run(torch, ctx, signals, sg.WANT_STAT)
    assert ctx.counters()["n_kernel_launches"] == 3
    names = [name for name, _, _ in ctx.stage_times()]
    assert names == ["stat_pa_moments", "stat_pa_median"], names
    both, _, _ = device_run(torch, ctx, signals, sg.WANT_STAT | sg.WANT_EVENTS)
    assert np.array_equal(bits(both), bits(stat))
    names = [name for name, _, _ in ctx.stage_times()]
    assert names[:2] == ["stat_pa_moments", "stat_pa_median"] and "pa_prefix" in names, names
    host = ctx.run_pa(signals, want=sg.WANT_STAT)
    assert ctx.counters()["n_kernel_launches"] == 3
    assert np.array_equal(bits(host.stat), bits(stat))
    check_ref(stat, signals, "stat only")


@pytest.mark.parametrize("rna", [0, 1])
def test_events_with_stat_are_events_alone(torch, ctx, rna):
    signals = arbitrary_signals(rna)
    alone = ctx.run_pa(signals, rna=rna, want=sg.WANT_EVENTS)
    both = ctx.run_pa(signals, rna=rna, want=sg.WANT_EVENTS | sg.WANT_STAT)
    assert_same_events(both, alone)
    assert np.array_equal(both.seq_order, alone.seq_order)
    check_ref(both.stat, signals, "events and stat")


def test_more_reads_than_the_grid(torch, ctx):
    """12,000 reads: more than the warps of the moments kernel's warp role (8 per CTA, 8 CTAs per SM), the CTAs of its
    CTA role and of the median kernels"""
    rng = np.random.default_rng(13)
    signals = [rng.normal(0, 3, int(n)).astype(F) for n in rng.integers(0, 700, 12_000)]
    for cta_min in (0, 1 << 31):
        ctx.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
        stats = all_paths(torch, ctx, signals)
        check_ref(stats["device"], signals, f"12,000 reads, cta_min {cta_min}")
        assert np.array_equal(bits(stats["host"]), bits(stats["device"]))


def test_stat_pa_helper(ctx):
    x = np.random.default_rng(14).normal(-1, 2, 3333).astype(F)
    got = sg.stat_pa(ctx, x)
    assert got.shape == (3,) and stat_mismatch(np.array([np.nan, got[0], np.nan, got[1], np.nan, got[2]], F),
                                               ref3(x)) == ""


PA = np.linspace(60.0, 90.0, 100).astype(np.float32)


def test_other_wants_are_refused(ctx):
    """with SGPU_F_PA_STAT a pA record computes EVENTS, STAT or both; every other product is refused on all three
    paths, and live entries stay events-only"""
    lib, h = ctx._lib, ctx._h
    for want in (sg.WANT_PA, sg.WANT_EVENTS | sg.WANT_PA, sg.WANT_STAT | sg.WANT_ENT, sg.WANT_ENT, sg.WANT_JNN,
                 sg.WANT_PREFIX, sg.WANT_SVBZD, sg.WANT_EVENTS | sg.WANT_SVBZD, 0):
        assert lib.sgpu_slot_reset(h, 0, 0) == 0
        assert lib.sgpu_slot_add_read_pa(h, 0, PA.ctypes.data, PA.size) == 0
        assert lib.sgpu_submit(h, 0, want) == E_INVAL, want
        with pytest.raises(sg.SgpuError) as e:
            ctx.run_device_pa(0, 0, 0, 0, 0, 0, want)
        assert e.value.code == E_INVAL, want
        with pytest.raises(sg.SgpuError) as e:
            ctx.run_device_pa_at(0, 0, 0, 0, 0, 8, 0, want)
        assert e.value.code == E_INVAL, want
    ctx.submit(0, sg.WANT_EVENTS | sg.WANT_STAT)
    res = ctx.wait(0, sg.WANT_EVENTS | sg.WANT_STAT)
    assert res.events(0).n >= 1 and stat_mismatch(res.stat[0], ref3(PA)) == ""
    with sg.Context(device=0, max_samples=4096, max_reads=8, flags=sg.F_PA_STAT) as c:
        c.live_open(2)
        assert c._lib.sgpu_slot_reset(c._h, 0, 0) == 0
        assert c._lib.sgpu_slot_add_live_pa(c._h, 0, 0, sg.LIVE_START | sg.LIVE_END, PA.ctypes.data, 100) == 0
        assert c._lib.sgpu_submit(c._h, 0, sg.WANT_STAT) == E_INVAL
        assert c._lib.sgpu_submit(c._h, 0, sg.WANT_EVENTS | sg.WANT_STAT) == E_INVAL


@pytest.mark.parametrize("flags", [0, sg.F_PA_STAT])
def test_wants_of_pa_slots_by_flag(torch, flags):
    """every want of a slot of pA records: EVENTS always, STAT and EVENTS | STAT only in a context opened with
    SGPU_F_PA_STAT; the device entries follow the same rule"""
    allowed = {sg.WANT_EVENTS} | ({sg.WANT_STAT, sg.WANT_EVENTS | sg.WANT_STAT} if flags else set())
    with sg.Context(device=0, max_samples=4096, max_reads=8, flags=flags) as c:
        lib, h = c._lib, c._h
        for want in range(128):
            assert lib.sgpu_slot_reset(h, 0, 0) == 0
            assert lib.sgpu_slot_add_read_pa(h, 0, PA.ctypes.data, PA.size) == 0
            rc = lib.sgpu_submit(h, 0, want)
            if want in allowed:
                assert rc == 0, want
                assert lib.sgpu_wait(h, 0, C.byref(_sl.Result())) == 0, want
            else:
                assert rc == E_INVAL, want
                assert lib.sgpu_wait(h, 0, C.byref(_sl.Result())) == E_STATE, want
        flat, off, lens = layout([PA])
        dev = torch.device("cuda:0")
        d_pa, d_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
        d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
        torch.cuda.synchronize()
        for want in (sg.WANT_STAT, sg.WANT_EVENTS | sg.WANT_STAT):
            span = int(off[-1])
            runs = (lambda: c.run_device_pa(d_pa.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), 1, span, 0, want),
                    lambda: c.run_device_pa_at(d_pa.data_ptr(), len(flat), d_off.data_ptr(), d_len.data_ptr(), 1, span,
                                               0, want))
            for run in runs:
                if flags:
                    run()
                    torch.cuda.synchronize()
                    assert c.counters()["status"] == 0
                else:
                    with pytest.raises(sg.SgpuError) as e:
                        run()
                    assert e.value.code == E_INVAL, want

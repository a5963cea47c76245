"""The svb-zd encoder on the GPU (SGPU_WANT_SVBZD on host slots, sgpu_encode_svbzd_device): every stream must equal,
byte for byte, what the reference's slow5lib writes (sha256 of its streams in tests/golden/ref_outputs.json, its
streams in svbzd_golden.npz, and the oracle's restatement of its encoder), the layout must feed the decoder unchanged,
and asking for the streams must change no other product."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import _refcases
from _oracle import Oracle
import sigtk_b200 as sg
from sigtk_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_OUT = json.load(open(os.path.join(G, "ref_outputs.json")))
E_INVAL, E_TOOBIG, E_STATE = -1, -5, -6
ALL_BUT_SVBZD = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX  # 63


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 26, max_reads=16384) as c:
        c.live_open(4)
        yield c


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def layout(raws):
    """the flat int16 array of `raws` with every read_off a multiple of ALIGN, read_off, read_len"""
    lens = np.array([len(r) for r in raws], np.int64)
    off = np.zeros(len(raws) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(max(int(off[-1]), 8), np.int16)
    for r, x in enumerate(raws):
        flat[off[r]:off[r] + lens[r]] = x
    return flat, off, lens


def host_encode(ctx, raws, slot=0):
    """-> the streams of a host slot of int16 records, and the slot's (comp_off, comp_len, bytes)"""
    res = ctx.run([(r, 8192.0, 0.0, 1.0) for r in raws], want=sg.WANT_SVBZD, slot=slot)
    return res.svbzd, slot_svb(ctx, slot, len(raws))


def slot_svb(ctx, slot, n):
    sv = sg._lib.SvbResult()
    assert ctx._lib.sgpu_slot_svbzd(ctx._h, slot, C.byref(sv)) == 0
    comp_off = np.ctypeslib.as_array(C.cast(sv.comp_off, C.POINTER(C.c_uint64)), shape=(n + 1,)).copy()
    comp_len = np.ctypeslib.as_array(C.cast(sv.comp_len, C.POINTER(C.c_uint32)), shape=(max(n, 1),))[:n].copy()
    assert int(sv.n_bytes) == int(comp_off[n])
    buf = (np.ctypeslib.as_array(C.cast(sv.bytes, C.POINTER(C.c_uint8)), shape=(int(sv.n_bytes),)).copy()
           if sv.n_bytes else np.empty(0, np.uint8))
    return comp_off, comp_len, buf


def device_encode(torch, ctx, raws):
    """sgpu_encode_svbzd_device on device copies of `raws`; -> (streams, (comp_off, comp_len, bytes), the result's
    device pointers, the device input arrays)"""
    flat, off, lens = layout(raws)
    arrs = [torch.from_numpy(x).cuda() for x in (flat, off, lens.astype(np.int32))]
    torch.cuda.synchronize()
    res = ctx.encode_svbzd_device(arrs[0].data_ptr(), arrs[1].data_ptr(), arrs[2].data_ptr(), len(raws), int(off[-1]),
                                  torch.cuda.current_stream().cuda_stream)
    n = len(raws)
    comp_off = ctx.d2h(res.comp_off, np.uint64, n + 1)  # (synchronises the device)
    comp_len = ctx.d2h(res.comp_len, np.uint32, n)
    buf = ctx.d2h(res.bytes, np.uint8, int(comp_off[n]))
    assert ctx.counters()["status"] == 0
    return streams_of(comp_off, comp_len, buf), (comp_off, comp_len, buf), res, arrs


def streams_of(comp_off, comp_len, buf):
    return [buf[int(o):int(o) + int(n)] for o, n in zip(comp_off[:-1], comp_len)]


def check_layout(comp_off, comp_len, buf):
    """streams on 16-byte boundaries, back to back, zeros between them; comp_off[n] = the bytes"""
    ends = comp_off[:-1] + comp_len.astype(np.uint64)
    assert comp_off[0] == 0 and np.all(comp_off % 16 == 0)
    assert np.array_equal(comp_off[1:], (ends + 15) // 16 * 16)
    assert int(comp_off[-1]) == len(buf)
    pad = np.zeros(len(buf), bool)
    for e, nxt in zip(ends, comp_off[1:]):
        pad[int(e):int(nxt)] = True
    assert not np.any(buf[pad])


def both_paths(torch, ctx, raws):
    """the streams of `raws` through a host slot and through sgpu_encode_svbzd_device, layouts checked"""
    h, hl = host_encode(ctx, raws)
    d, dl, _, _ = device_encode(torch, ctx, raws)
    check_layout(*hl)
    check_layout(*dl)
    return {"host": h, "device": d}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- the reference's bytes -------------------------------------------------------------------------------------------
def test_reference_streams_by_sha256(torch, ctx):
    for name, raws in (("svbzd_grid", _refcases.svbzd_grid()), ("svbzd_reads", _refcases.svbzd_reads())):
        assert len(raws) == len(REF_OUT[name])
        for path, streams in both_paths(torch, ctx, raws).items():
            assert [sha(s) for s in streams] == REF_OUT[name], (name, path)


def test_golden_streams_written_by_slow5lib(torch, ctx):
    d = np.load(os.path.join(G, "svbzd_golden.npz"))
    names = [k[4:] for k in d.files if k.startswith("raw_") and k != "raw_wide_codes"]  # (wide_codes: decode-only)
    assert len(names) >= 9
    for path, streams in both_paths(torch, ctx, [d["raw_" + k] for k in names]).items():
        for k, s in zip(names, streams):
            assert np.array_equal(s, d["svb_" + k]), (k, path)


# ---- edges against the oracle ---------------------------------------------------------------------------------------
def edge_reads():
    rng = np.random.default_rng(7)
    out = []
    for n in (0, 1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 2047, 2048, 2049, 4097):
        for scale in (3, 200, 40000):
            out.append(np.clip(np.cumsum(rng.integers(-scale, scale + 1, n)), -32768, 32767).astype(np.int16))
    # deltas on every code boundary: z = 255 / 256 (d = -128 / 128) and 65,535 / 65,536 (d = -32,768 / 32,768), and
    # d = 127, -127, 32,767, -32,767 beside them
    for d in (127, 128, -127, -128, 32767, 32768, -32767, -32768):
        walk = [0]
        for k in range(3000):
            nxt = walk[-1] + (d if k % 2 == 0 else -d)
            walk.append(nxt)
        base = -16384 if d > 0 else 16383
        out.append((np.array(walk[1:], np.int64) + base).astype(np.int16))
    out.append(np.tile(np.array([-32768, 32767], np.int16), 2500))  # every value 3 bytes
    out.append(np.full(5000, 1234, np.int16))                       # constant
    out.append(np.concatenate([[32767], rng.integers(-5, 6, 2000)]).astype(np.int16))  # raw[-1] = 0: a 2-byte first value
    out.append(np.concatenate([[-32768], np.full(40, -32768)]).astype(np.int16))        # a 3-byte first value
    return out


def test_edges_equal_the_oracle(torch, ctx, orc):
    raws = edge_reads()
    # empty reads between non-empty ones
    raws = [x for r in raws for x in (r, np.zeros(0, np.int16))]
    for path, streams in both_paths(torch, ctx, raws).items():
        for r, (s, raw) in enumerate(zip(streams, raws)):
            assert np.array_equal(s, orc.svbzd_encode(raw)), (path, r, len(raw))


def test_code_boundaries_are_hit(orc):
    """the edge reads do take values of 1, 2 and 3 bytes on both sides of each code boundary"""
    z = []
    for raw in edge_reads():
        x = np.concatenate([[0], raw.astype(np.int64)])
        d = (x[1:] - x[:-1]).astype(np.int32)
        z.append(((d.astype(np.uint32) << np.uint32(1)) ^ (d >> 31).astype(np.uint32)))
    z = set(np.concatenate(z).tolist())
    assert {254, 255, 256, 65534, 65535, 65536, 131070} <= z


def test_per_record_convenience(ctx, orc):
    raw = synth.make_read(3, 12345, seed=4)[0]
    assert np.array_equal(sg.svbzd_encode(ctx, raw), orc.svbzd_encode(raw))


# ---- scale -----------------------------------------------------------------------------------------------------------
def test_ten_thousand_reads_and_a_long_read(torch, ctx, orc):
    """enough blocks that every block loop runs more than once (148 SMs x 64 warps), and a 2,000,000-sample read"""
    raws = [rd[0] for rd in synth.make_reads(10000, mean=3000.0, seed=23)]
    raws.insert(4321, synth.make_read(1, 2_000_000, seed=24)[0])
    want = [orc.svbzd_encode(r) for r in raws]
    for path, streams in both_paths(torch, ctx, raws).items():
        assert len(streams) == len(want)
        for r, (s, w) in enumerate(zip(streams, want)):
            assert np.array_equal(s, w), (path, r, len(raws[r]))


# ---- round trip ------------------------------------------------------------------------------------------------------
def test_device_output_feeds_the_decoder(torch, ctx):
    raws = [rd[0] for rd in synth.make_reads(300, mean=20000.0, seed=31)] + edge_reads()
    _, (comp_off, comp_len, buf), res, arrs = device_encode(torch, ctx, raws)
    flat, off, lens = layout(raws)
    out = torch.zeros(len(flat), dtype=torch.int16, device="cuda")
    n_blocks = int(((lens + 1023) // 1024).sum())
    ctx.decode_svbzd_device(res.bytes, int(comp_off[-1]), res.comp_off, res.comp_len, arrs[1].data_ptr(),
                            arrs[2].data_ptr(), len(raws), n_blocks, out.data_ptr(),
                            torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert ctx.counters()["status"] == 0
    got = out.cpu().numpy()
    for r in range(len(raws)):
        assert np.array_equal(got[off[r]:off[r] + lens[r]], raws[r]), r


@pytest.mark.parametrize("rna", [0, 1])
def test_streams_into_an_svbzd_slot_give_the_same_events(torch, ctx, rna):
    reads = synth.make_reads(60, mean=25000.0, seed=41 + rna, rna=bool(rna))
    want = sg.WANT_EVENTS | sg.WANT_PA
    a = ctx.run(reads, rna=rna, want=want | sg.WANT_SVBZD)
    dstreams = device_encode(torch, ctx, [rd[0] for rd in reads])[0]
    for streams in (a.svbzd, dstreams):
        b = ctx.run_svbzd([(s, rd[1], rd[2], rd[3]) for s, rd in zip(streams, reads)], rna=rna, want=want)
        assert np.array_equal(a.ev_off, b.ev_off) and np.array_equal(a.ev_start, b.ev_start)
        assert np.array_equal(a.ev_mean.view(np.uint32), b.ev_mean.view(np.uint32))
        assert np.array_equal(a.ev_stdv.view(np.uint32), b.ev_stdv.view(np.uint32))
        for x, y in zip(a.pa, b.pa):  # the samples themselves, through pA
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


# ---- svb-zd slots ----------------------------------------------------------------------------------------------------
def test_svbzd_slot_returns_its_input_streams(ctx, orc):
    d = np.load(os.path.join(G, "svbzd_golden.npz"))
    names = [k[4:] for k in d.files if k.startswith("raw_")]
    raws = [d["raw_" + k] for k in names] + _refcases.svbzd_reads()
    streams = [d["svb_" + k] for k in names] + [orc.svbzd_encode(r) for r in _refcases.svbzd_reads()]
    res = ctx.run_svbzd([(s, 1.0, 0.0, 1.0) for s in streams], want=sg.WANT_SVBZD | sg.WANT_STAT)
    check_layout(*slot_svb(ctx, 0, len(streams)))
    for k, (got, s, raw) in enumerate(zip(res.svbzd, streams, raws)):
        if k < len(names) and names[k] == "wide_codes":  # hand-made 4-byte codes: back in canonical form
            assert not np.array_equal(got, s)
            assert np.array_equal(got, orc.svbzd_encode(raw))
        else:
            assert np.array_equal(got, s), k


# ---- no side effects -------------------------------------------------------------------------------------------------
def same_products(a, b):
    assert np.array_equal(a.ev_off, b.ev_off) and np.array_equal(a.ev_start, b.ev_start)
    for x, y in ((a.ev_mean, b.ev_mean), (a.ev_stdv, b.ev_stdv), (a.stat, b.stat), (a.prefix_stat, b.prefix_stat)):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    assert np.array_equal(a.ent.view(np.uint64), b.ent.view(np.uint64))
    assert np.array_equal(a.prefix_pos, b.prefix_pos)
    assert np.array_equal(a.seq_order, b.seq_order) and np.array_equal(a.fixups, b.fixups)
    assert len(a.jnn) == len(b.jnn) and all(np.array_equal(x, y) for x, y in zip(a.jnn, b.jnn))
    assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a.pa, b.pa))


@pytest.mark.parametrize("rna", [0, 1])
def test_other_products_do_not_change(ctx, orc, rna):
    reads = synth.make_reads(80, mean=30000.0, seed=51 + rna, rna=bool(rna))
    reads += [synth.make_read_cb(k, n, seed=5) for k, n in enumerate((0, 1, 7, 2001))]
    a = ctx.run(reads, rna=rna, want=ALL_BUT_SVBZD)
    b = ctx.run(reads, rna=rna, want=ALL_BUT_SVBZD | sg.WANT_SVBZD, slot=1)
    same_products(a, b)
    for s, rd in zip(b.svbzd, reads):
        assert np.array_equal(s, orc.svbzd_encode(rd[0]))
    streams = [orc.svbzd_encode(rd[0]) for rd in reads]  # and on an svb-zd slot
    c = ctx.run_svbzd([(s, rd[1], rd[2], rd[3]) for s, rd in zip(streams, reads)], rna=rna,
                      want=ALL_BUT_SVBZD | sg.WANT_SVBZD)
    same_products(a, c)
    assert all(np.array_equal(x, y) for x, y in zip(c.svbzd, streams))


def test_two_slots_in_flight_keep_their_streams(ctx, orc):
    ra = [rd[0] for rd in synth.make_reads(50, mean=20000.0, seed=61)]
    rb = [rd[0] for rd in synth.make_reads(70, mean=9000.0, seed=62)]
    ctx.fill(0, [(r, 8192.0, 0.0, 1.0) for r in ra], 0)
    ctx.fill(1, [(r, 8192.0, 0.0, 1.0) for r in rb], 0)
    ctx.submit(0, sg.WANT_SVBZD | sg.WANT_EVENTS)
    ctx.submit(1, sg.WANT_SVBZD)
    b = ctx.wait(1, sg.WANT_SVBZD)
    a = ctx.wait(0, sg.WANT_SVBZD | sg.WANT_EVENTS)
    for res, raws in ((a, ra), (b, rb)):
        assert len(res.svbzd) == len(raws)
        for s, r in zip(res.svbzd, raws):
            assert np.array_equal(s, orc.svbzd_encode(r))
    # still there after the other slot's next batch
    ctx.run([(r, 8192.0, 0.0, 1.0) for r in rb[:5]], want=sg.WANT_SVBZD, slot=1)
    comp_off, comp_len, buf = slot_svb(ctx, 0, len(ra))
    assert all(np.array_equal(s, orc.svbzd_encode(r)) for s, r in zip(streams_of(comp_off, comp_len, buf), ra))


def test_empty_slot_and_empty_reads(torch, ctx):
    ctx._check(ctx._lib.sgpu_slot_reset(ctx._h, 0, 0))
    ctx.submit(0, sg.WANT_SVBZD)
    assert ctx.wait(0, sg.WANT_SVBZD).svbzd == []
    assert slot_svb(ctx, 0, 0)[0].tolist() == [0]
    for path, streams in both_paths(torch, ctx, [np.zeros(0, np.int16)] * 3).items():
        assert [s.tolist() for s in streams] == [[0, 0, 0, 0]] * 3, path


# ---- refusals --------------------------------------------------------------------------------------------------------
def test_refusals(torch, ctx):
    lib, h = ctx._lib, ctx._h
    raw = synth.make_read(1, 3000, seed=2)[0]
    ctx.fill_pa(0, [raw.astype(np.float32)], 0)  # pA records
    assert lib.sgpu_submit(h, 0, sg.WANT_SVBZD) == E_INVAL
    assert lib.sgpu_submit(h, 0, sg.WANT_SVBZD | sg.WANT_EVENTS) == E_INVAL
    ctx.live_fill(0, [(0, sg.LIVE_START, raw, 8192.0, 0.0, 1.0)])  # int16 live entries
    assert lib.sgpu_submit(h, 0, sg.WANT_SVBZD | sg.WANT_EVENTS) == E_INVAL
    ctx.live_fill_pa(0, [(1, sg.LIVE_START, raw.astype(np.float32))])  # pA live entries
    assert lib.sgpu_submit(h, 0, sg.WANT_SVBZD) == E_INVAL
    ctx.fill(0, [(raw, 8192.0, 0.0, 1.0)], 0)
    for want in (128, 129, 255, 1 << 31):  # bits above 127
        assert lib.sgpu_submit(h, 0, want) == E_INVAL
    # sgpu_slot_svbzd: before the wait, without the bit, after a reset
    sv = sg._lib.SvbResult()
    ctx.submit(0, sg.WANT_SVBZD)
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == E_STATE
    ctx.wait(0, sg.WANT_SVBZD)
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == 0 and sv.n_bytes > 0
    ctx.submit(0, sg.WANT_STAT)
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == E_STATE
    ctx.wait(0, sg.WANT_STAT)
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == E_STATE
    ctx.run([(raw, 8192.0, 0.0, 1.0)], want=sg.WANT_SVBZD)
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == 0
    ctx._check(lib.sgpu_slot_reset(h, 0, 0))
    assert lib.sgpu_slot_svbzd(h, 0, C.byref(sv)) == E_STATE
    # bit 64 in sgpu_run_device
    flat, off, lens = layout([raw])
    arrs = [torch.from_numpy(x).cuda() for x in (flat, off, lens.astype(np.int32), np.zeros(1, np.float32),
                                                 np.ones(1, np.float32))]
    torch.cuda.synchronize()
    for want in (sg.WANT_SVBZD, sg.WANT_SVBZD | sg.WANT_EVENTS):
        with pytest.raises(sg.SgpuError) as e:
            ctx.run_device(*[a.data_ptr() for a in arrs], 1, int(off[-1]), 0, want)
        assert e.value.code == E_INVAL
    # a device batch the context cannot hold
    with pytest.raises(sg.SgpuError) as e:
        ctx.encode_svbzd_device(arrs[0].data_ptr(), arrs[1].data_ptr(), arrs[2].data_ptr(), 1, ctx.max_samples + 64)
    assert e.value.code == E_INVAL


def test_device_span_over_the_stream_limit_is_refused(torch):
    """a context of more than 1.32 G samples (no host slots): a span past the limit is SGPU_E_TOOBIG before any kernel
    runs; the slot path's per-read check uses the same function (test_svbzd_limit.py checks its bound on the CPU)"""
    limit = 1_321_528_397
    span = (limit + 8) // 8 * 8
    with sg.Context(device=0, max_samples=span, max_reads=4, n_slots=0, flags=sg.F_NO_HOST_SLOTS) as c:
        dummy = torch.zeros(16, dtype=torch.int64, device="cuda")
        with pytest.raises(sg.SgpuError) as e:
            c.encode_svbzd_device(dummy.data_ptr(), dummy.data_ptr(), dummy.data_ptr(), 1, span)
        assert e.value.code == E_TOOBIG

"""GPU parity of the svb-zd decoder (sigtk_b200/csrc/svbzd.cu) through the C-ABI: samples decoded in HBM from the
streams slow5lib stores in BLOW5 records must equal the reference's own decode (golden streams written by the
reference's slow5lib, streams checked byte for byte against the reference's by their sha256, the oracle), and the
whole path (streams in -> events / pA / stat out) must equal the path fed with decoded records."""
import hashlib
import json
import os

import numpy as np
import pytest

import sigtk_b200 as sg
import _refcases
from _oracle import Oracle
from sigtk_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 23, max_reads=4096) as c:
        yield c


def decode_on_gpu(ctx, streams):
    """the decoded samples of every stream: the stat path returns raw_median etc., but the samples themselves are
    read back through pA with offset 0, range == digitisation (pA == raw exactly)"""
    res = ctx.run_svbzd([(s, 1.0, 0.0, 1.0) for s in streams], want=sg.WANT_PA)
    return [p.astype(np.int64) for p in res.pa]


def test_golden_streams(ctx):
    d = np.load(os.path.join(G, "svbzd_golden.npz"))
    names = [k[4:] for k in d.files if k.startswith("raw_")]
    got = decode_on_gpu(ctx, [d["svb_" + k] for k in names])
    for k, g in zip(names, got):
        assert np.array_equal(g, d["raw_" + k].astype(np.int64)), k


@pytest.mark.parametrize("scale", [3, 200, 40000])
def test_ragged_lengths_and_code_mixes(ctx, orc, scale):
    """lengths around the lane (32), block (1024) and key-word (16) sizes; 1-, 2- and 3-byte values"""
    rng = np.random.default_rng(scale)
    raws = []
    for n in [0, 1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 2047, 2048, 2049, 4097, 33333,
              200001]:
        raws.append(np.clip(np.cumsum(rng.integers(-scale, scale + 1, n)), -32768, 32767).astype(np.int16))
    streams = [orc.svbzd_encode(r) for r in raws]
    for g, r in zip(decode_on_gpu(ctx, streams), raws):
        assert np.array_equal(g, r.astype(np.int64)), len(r)


def test_wraparound(ctx, orc):
    """deltas that overflow int16 and a running value that wraps in 32 bits exactly like the reference's int32 prev"""
    raw = np.tile(np.array([32767, -32768], np.int16), 3000)
    stream = orc.svbzd_encode(raw)
    assert np.array_equal(decode_on_gpu(ctx, [stream])[0], raw.astype(np.int64))


def test_streams_written_by_reference_slow5lib(ctx, orc):
    """the streams the reference's slow5lib writes for 24 synthetic reads (each made here and checked against the
    sha256 of the reference's bytes in tests/golden/ref_outputs.json) decode on the GPU to the reads"""
    raws = _refcases.svbzd_reads()
    want = json.load(open(os.path.join(G, "ref_outputs.json")))["svbzd_reads"]
    streams = [orc.svbzd_encode(r) for r in raws]
    assert [hashlib.sha256(s.tobytes()).hexdigest() for s in streams] == want
    for g, r in zip(decode_on_gpu(ctx, streams), raws):
        assert np.array_equal(g, r.astype(np.int64))


@pytest.mark.parametrize("rna", [0, 1])
def test_whole_path_from_streams_equals_decoded_records(ctx, orc, rna):
    reads = synth.make_reads(40, mean=25000.0, seed=17 + rna, rna=bool(rna))
    want = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT
    a = ctx.run(reads, rna=rna, want=want)
    b = ctx.run_svbzd([(orc.svbzd_encode(r[0]), r[1], r[2], r[3]) for r in reads], rna=rna, want=want)
    assert np.array_equal(a.ev_off, b.ev_off) and np.array_equal(a.ev_start, b.ev_start)
    assert np.array_equal(a.ev_mean.view(np.uint32), b.ev_mean.view(np.uint32))
    assert np.array_equal(a.ev_stdv.view(np.uint32), b.ev_stdv.view(np.uint32))
    assert np.array_equal(a.stat.view(np.uint32), b.stat.view(np.uint32))
    for x, y in zip(a.pa, b.pa):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    st, ln, mn, sd = orc.events(*reads[3], rna=rna)
    assert np.array_equal(b.events(3).start, st)


def test_malformed_streams_are_reported(ctx, orc):
    raw = synth.make_read(1, 5000, seed=2)[0]
    st = orc.svbzd_encode(raw)
    with pytest.raises(sg.SgpuError) as e:   # header says more values than the bytes can hold
        ctx.run_svbzd([(st[: 4 + (len(raw) + 3) // 4 + 10], 1.0, 0.0, 1.0)], want=sg.WANT_STAT)
    assert e.value.code == -9
    with pytest.raises(sg.SgpuError) as e:   # one byte too many: the keys do not account for it (slow5_press.c:1103)
        ctx.run_svbzd([(np.concatenate([st, st[-1:]]), 1.0, 0.0, 1.0)], want=sg.WANT_STAT)
    assert e.value.code == -9
    with pytest.raises(sg.SgpuError) as e:   # truncated data
        ctx.run_svbzd([(st[:-3], 1.0, 0.0, 1.0)], want=sg.WANT_STAT)
    assert e.value.code == -9
    ok = ctx.run_svbzd([(st, 1.0, 0.0, 1.0)], want=sg.WANT_STAT)  # the context is usable afterwards
    assert ok.n_reads == 1


def test_mixing_records_and_streams_is_refused(ctx, orc):
    raw = synth.make_read(1, 3000, seed=2)[0]
    ctx.fill(0, [(raw, 8192.0, 3.0, 1400.0)], 0)
    rc = ctx._lib.sgpu_slot_add_read_svbzd(ctx._h, 0, orc.svbzd_encode(raw).ctypes.data, 10, 1.0, 0.0, 1.0)
    assert rc == -6
    ctx._lib.sgpu_slot_reset(ctx._h, 0, 0)

"""GPU parity tests at batch sizes where every kernel's grid-stride loop runs more than once.

Every kernel caps its grid (a multiple of the SM count) and loops, so a warp or CTA whose work runs past the grid takes
a second and third item: prefetches of the next tile, shared arrays reused behind a __syncwarp, per-read values that
must be reset between reads. Those passes only happen on batches of production size (tens of millions of samples,
thousands of reads). Here such batches are checked read by read against the CPU oracle with the exactness of the other
parity tests: bits for events, pA, stat, jnn and prefix, 1e-12 absolute for ent.

Each test first asserts its premise -- that the batch is larger than the single-pass capacity of the kernels it is
about, computed from the launch shapes below and the device's SM count -- so that a change of a launch shape fails
loudly instead of quietly testing nothing. The premises are printed (run with -s to see them).

Also here: contexts of production size whose sequential-order scratch is an eighth of the batch (SGPU_E_SCRATCH),
the long detector's job list past the grid and past its capacity, a batch that fills its context exactly, and the
adaptor parameters of RNA004 pores (SGPU_PARAM_PORE)."""
import concurrent.futures as cf
import contextlib
import os
import time

import numpy as np
import pytest

from _oracle import Oracle
import sigtk_b200 as sg
from sigtk_b200 import _lib as _sl
from sigtk_b200 import synth
from test_gpu_parity import _fuzz_read
from test_gpu_prefix import adaptor_read
from test_host_walk import glitch_read

pytestmark = pytest.mark.gpu

ALL6 = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
F_FULL_SEQ_SCRATCH = 8          # SGPU_F_FULL_SEQ_SCRATCH (include/sigtk_b200.h)
ENT_TOL = 1e-12
TINY_LENS = [1, 2, 5, 6, 7, 8, 9, 11, 12, 13, 15, 16, 17, 27, 28, 29, 31, 32, 33, 63, 64, 65, 199, 200, 201, 255, 256,
             257, 1023, 1024, 1025, 4095, 4096, 4097]


# ---- launch shapes: the work one launch covers before its grid-stride loop comes round again --------------------------
def single_pass(sm):
    """items one wave of the grid takes, per kernel, for `sm` streaming multiprocessors"""
    return {
        # emit.cu:337  grid_cap(n_wt, EWARPS, sm * EMIT_GRID): 64 CTAs/SM x 4 warps x 1,024-sample warp tiles
        "emit_events_samples": sm * 64 * 4 * 1024,
        # generic.cu:491  grid_cap(.., 256, sm * 16): 8 warps x 32 lanes x PA_IT (8) groups of 8 samples
        "pa_samples": sm * 16 * 8 * 2048,
        # svbzd.cu:217  grid_cap(max_blocks, SVB_WARPS, sm * 16): 4 warps x 1,024-value blocks
        "svbzd_samples": sm * 16 * 4 * 1024,
        # fast.cu:145  grid_cap(n_tiles * 32, 256, sm * 8): 8 warps x 2,048-sample tiles
        "count_tile_bits_samples": sm * 8 * 8 * 2048,
        # walk.cu:422  grid_cap(max_interior + n_reads, 256, sm * 8): a thread per chunk boundary
        "verify_chunks_items": sm * 8 * 256,
        # stat.cu:299-302  warp role: <= sm * 8 CTAs x 8 warps, a warp per read; CTA role: sm * 2 CTAs
        "stat_warp_reads": sm * 8 * 8,
        "stat_cta_reads": sm * 2,
        # stat.cu:313-314  stat_median_kernel<1024>: sm * 2 CTAs; <256>: sm * 8 CTAs, a CTA per read
        "stat_median1024_reads": sm * 2,
        "stat_median256_reads": sm * 8,
        # prefix.cu:312-318  prefix_walk_kernel: sm * 16 CTAs x 4 warps, a warp per read; prefix_median_kernel: sm * 8
        "prefix_walk_reads": sm * 16 * 4,
        "prefix_median_reads": sm * 8,
        # ent.cu:209  a CTA per read, sm * 4 CTAs
        "ent_reads": sm * 4,
        # generic.cu:468-485  gen_prefix / gen_detect / gen_emit: sm * 8 CTAs x 4 warps; gen_tstat: sm * 8 CTAs
        "gen_warp_reads": sm * 8 * 4,
        "gen_tstat_reads": sm * 8,
        # walk.cu:414-415  long_jobs_kernel: RNA a warp per life (sm * 16 CTAs x 4 warps), DNA a thread (sm * 4 x 128)
        "long_jobs_rna": sm * 16 * 4,
        "long_jobs_dna": sm * 4 * 128,
    }


def premise(what, value, bound, factor=1.0):
    """the test is only about what it claims when value > factor * bound"""
    msg = f"premise: {what} {value:.4g} > {factor * bound:.4g} ({factor:g} x {bound:.4g})"
    print(msg)
    assert value > factor * bound, msg


def walk_chunk_len(span, n_reads, rna, sm, forced=0):
    """walk.cu:355-371 (the chunk length the walker picks for a batch)"""
    lmin = 512 if rna else 128
    want = sm * (2048 if rna else 384)
    L = 4096 if rna else 1024
    while L > lmin and span // L < want:
        L >>= 1
    if n_reads:
        per_read = span // n_reads // 12 // 128 * 128
        if per_read < L:
            L = per_read if per_read > lmin else lmin
    if forced >= lmin and forced % 32 == 0:
        L = forced
    return L


def verify_items(lens, L):
    """work items of verify_chunks_kernel: interior chunks of every read, then the last chunk of every read"""
    nch = (np.asarray(lens, np.int64) + L - 1) // L
    return int(np.maximum(nch - 2, 0).sum()) + len(lens)


def span_of(reads):
    return int(sum((len(r[0]) + 7) // 8 * 8 for r in reads))


@pytest.fixture(scope="module")
def sm():
    torch = pytest.importorskip("torch")
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def cap(sm):
    return single_pass(sm)


@pytest.fixture(scope="module")
def orc():
    return Oracle()


class Contexts:
    """One context at a time: asking for another size closes the previous one first, so the file never holds more
    than one context's memory (a few GB) on a shared device."""

    def __init__(self):
        self.key, self.ctx = None, None

    def get(self, max_samples, max_reads, flags=sg.F_DEFAULT):
        key = (max_samples, max_reads, flags)
        if key != self.key:
            self.close()
            self.ctx = sg.Context(device=0, max_samples=max_samples, max_reads=max_reads, flags=flags)
            self.key = key
        return self.ctx

    def close(self):
        if self.ctx is not None:
            self.ctx.close()
        self.key, self.ctx = None, None


@pytest.fixture(scope="module")
def contexts():
    t0 = time.time()
    c = Contexts()
    yield c
    c.close()
    print(f"\ntest_gpu_waves: wall time {time.time() - t0:.1f} s")


@contextlib.contextmanager
def params(ctx, **kv):
    """context parameters (sgpu_set_param) for the duration of a block, restored to their defaults afterwards"""
    keys = {"chunk_len": (_sl.PARAM_CHUNK_LEN, 0), "warmup": (_sl.PARAM_WARMUP, 0), "thr_long": (_sl.PARAM_THR_LONG, 9.0),
            "stat_cta_min": (_sl.PARAM_STAT_CTA_MIN, 131072), "pore": (_sl.PARAM_PORE, 0)}
    for k, v in kv.items():
        ctx.set_param(keys[k][0], v)
    try:
        yield ctx
    finally:
        for k in kv:
            ctx.set_param(*keys[k])


def pmap(fn, items):
    """the oracle is independent per read and its ctypes calls release the GIL"""
    with cf.ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2)) as ex:
        return list(ex.map(fn, items))


def bits(a):
    return np.asarray(a).view(np.uint32) if np.asarray(a).dtype == np.float32 else np.asarray(a)


def read_mismatches(orc, res, reads, rna, want, r, pore=0):
    """what differs between the GPU's outputs for read r and the oracle's (empty list: nothing)"""
    rd, bad = reads[r], []
    if want & sg.WANT_EVENTS:
        st, ln, mn, sd = orc.events(*rd, rna=rna)
        ev = res.events(r)
        if not np.array_equal(ev.start, st):
            bad.append("event starts")
        elif not (np.array_equal(bits(ev.length), bits(ln)) and np.array_equal(bits(ev.mean), bits(mn))
                  and np.array_equal(bits(ev.stdv), bits(sd))):
            bad.append("event length / mean / stdv")
    if want & sg.WANT_PA and not np.array_equal(bits(res.pa[r]), bits(orc.pa(*rd))):
        bad.append("pA")
    if want & sg.WANT_STAT and not np.array_equal(bits(res.stat[r]), bits(orc.stat(*rd))):
        bad.append("stat")
    if want & sg.WANT_ENT and not np.allclose(res.ent[r], orc.ent(rd[0]), rtol=0, atol=ENT_TOL):
        bad.append("ent")
    if want & sg.WANT_JNN and not np.array_equal(res.jnn[r], orc.jnn(rd[0], rna)):
        bad.append("jnn")
    if want & sg.WANT_PREFIX:
        pos, pst = orc.adaptor_polya(*rd, rna=rna, pore=pore)
        got_pos, got_st = res.prefix_pos[r].astype(np.int64), res.prefix_stat[r]
        if not np.array_equal(got_pos, pos):
            bad.append(f"prefix positions {got_pos} != {pos}")
        elif (pos[1] > 0 and not np.array_equal(bits(got_st[:3]), bits(pst[:3]))) or \
                (pos[3] > 0 and not np.array_equal(bits(got_st[3:]), bits(pst[3:]))):
            bad.append("prefix statistics")
    return bad


def check_all(orc, res, reads, rna, want, pore=0):
    """every read against the oracle; on failure the message names the reads, their lengths and what differs"""
    found = pmap(lambda r: (r, read_mismatches(orc, res, reads, rna, want, r, pore)), range(len(reads)))
    bad = [(r, len(reads[r][0]), what) for r, what in found if what]
    assert not bad, f"{len(bad)} of {len(reads)} reads differ (read, length, what): {bad[:8]}"


def event_starts_at(orc, rd, rna, thr):
    return orc.event_starts(*rd, rna=rna, thr_long=thr)


# ---- the production-size batch shared by tests 1-4 -------------------------------------------------------------------
BIG_SAMPLES, BIG_READS = 1 << 27, 32768


@pytest.fixture(scope="module")
def big_reads():
    return make_big_reads()


def make_big_reads():
    """~20,000 ragged reads of 1-6,000 samples with the tiny and around-the-window lengths mixed in, 500 adaptor /
    poly-A reads of 20-40 k samples and 200 adversarial reads, shuffled so that every kind is spread over the batch"""
    rng = np.random.default_rng(2027)
    lens = rng.integers(1, 6001, 20000)
    lens[::500] = np.resize(TINY_LENS, lens[::500].shape)
    lens[250::500] = np.resize(TINY_LENS[::-1], lens[250::500].shape)
    reads = [synth.make_read(k, int(n), seed=4040) for k, n in enumerate(lens)]
    reads += [adaptor_read(k, int(n), seed=4041) for k, n in enumerate(rng.integers(20000, 40001, 500))]
    fz = np.random.default_rng(4042)
    reads += [_fuzz_read(fz, k) for k in range(200)]
    order = rng.permutation(len(reads))
    return [reads[i] for i in order]


def big_premises(reads, cap):
    span = span_of(reads)
    premise("span (samples) over emit_events_kernel's grid", span, cap["emit_events_samples"], 1.5)
    premise("span (samples) over count_tile_bits_kernel's grid", span, cap["count_tile_bits_samples"], 2.0)
    n = len(reads)
    premise("reads over stat_moments_kernel's warps", n, cap["stat_warp_reads"], 2.0)
    premise("reads over prefix_walk_kernel's warps", n, cap["prefix_walk_reads"], 2.0)
    premise("reads over stat_median_kernel<256>'s CTAs", n, cap["stat_median256_reads"], 2.0)
    premise("reads over prefix_median_kernel's CTAs", n, cap["prefix_median_reads"], 2.0)
    premise("reads over ent_kernel's CTAs", n, cap["ent_reads"], 2.0)


@pytest.mark.parametrize("rna", [0, 1])
def test_many_reads_every_product(contexts, orc, cap, big_reads, rna):
    """test 1: every product of every read of a batch that takes every per-read and per-tile kernel past its grid"""
    big_premises(big_reads, cap)
    ctx = contexts.get(BIG_SAMPLES, BIG_READS)
    res = ctx.run(big_reads, rna=rna, want=ALL6)
    check_all(orc, res, big_reads, rna, ALL6)
    n_prefix = int((res.prefix_pos[:, 1] > 0).sum())
    print(f"rna={rna}: {int(res.ev_off[-1])} events, {n_prefix} adaptors, {int(res.seq_order.sum())} sequential-order reads")
    assert n_prefix >= 100


def test_pa_kernel_past_its_grid(contexts, orc, cap, big_reads):
    """test 2: pA without events is stored by pa_kernel (not by the walker's fused store)"""
    premise("span (samples) over pa_kernel's grid", span_of(big_reads), cap["pa_samples"], 1.5)
    ctx = contexts.get(BIG_SAMPLES, BIG_READS)
    for want in (sg.WANT_PA, sg.WANT_PA | sg.WANT_STAT):
        check_all(orc, ctx.run(big_reads, rna=0, want=want), big_reads, 0, want)


@pytest.mark.parametrize("cta_min", [1024, 0])
def test_stat_cta_role_past_its_grid(contexts, orc, cap, big_reads, cta_min):
    """test 3: with STAT_CTA_MIN lowered thousands of reads take the CTA role of the moments kernels and
    stat_median_kernel<1024>, over their sm * 2 CTAs"""
    n_cta = sum(1 for rd in big_reads if len(rd[0]) >= cta_min)
    premise(f"reads of >= {cta_min} samples over the CTA role's CTAs", n_cta, cap["stat_cta_reads"], 2.0)
    premise(f"reads of >= {cta_min} samples over stat_median_kernel<1024>'s CTAs", n_cta, cap["stat_median1024_reads"], 2.0)
    ctx = contexts.get(BIG_SAMPLES, BIG_READS)
    with params(ctx, stat_cta_min=cta_min):
        res = ctx.run(big_reads, rna=0, want=sg.WANT_STAT | sg.WANT_JNN)
    check_all(orc, res, big_reads, 0, sg.WANT_STAT | sg.WANT_JNN)


def test_svbzd_past_its_grid(contexts, orc, cap, big_reads):
    """test 4: the same batch as svb-zd streams decoded in HBM gives the same bits in every output; a copy with
    range == digitisation and offset 0 (pA = raw) shows the decoded samples themselves"""
    premise("span (samples) over the svb-zd kernels' grid", span_of(big_reads), cap["svbzd_samples"], 1.5)
    ctx = contexts.get(BIG_SAMPLES, BIG_READS)
    streams = pmap(lambda rd: orc.svbzd_encode(rd[0]), big_reads)
    raw = ctx.run(big_reads, rna=1, want=ALL6)
    res = ctx.run_svbzd([(s, rd[1], rd[2], rd[3]) for s, rd in zip(streams, big_reads)], rna=1, want=ALL6)
    assert np.array_equal(res.ev_off, raw.ev_off) and np.array_equal(res.ev_start, raw.ev_start)
    assert np.array_equal(bits(res.ev_mean), bits(raw.ev_mean)) and np.array_equal(bits(res.ev_stdv), bits(raw.ev_stdv))
    assert np.array_equal(bits(res.stat), bits(raw.stat)) and np.array_equal(res.ent, raw.ent)
    assert np.array_equal(res.prefix_pos, raw.prefix_pos) and np.array_equal(bits(res.prefix_stat), bits(raw.prefix_stat))
    assert np.array_equal(res.seq_order, raw.seq_order)
    for r in range(len(big_reads)):
        assert np.array_equal(bits(res.pa[r]), bits(raw.pa[r])), f"read {r}: pA differs"
        assert np.array_equal(res.jnn[r], raw.jnn[r]), f"read {r}: jnn differs"
    ident = ctx.run_svbzd([(s, 8192.0, 0.0, 8192.0) for s in streams], rna=0, want=sg.WANT_PA)
    for r, rd in enumerate(big_reads):
        assert np.array_equal(ident.pa[r], rd[0].astype(np.float32)), f"read {r}: decoded samples differ"


# ---- sequential-order kernels -----------------------------------------------------------------------------------------
def test_many_sequential_order_reads(contexts, orc, cap):
    """test 5: every read of a forced-generic batch walks the compacted work list of the sequential-order kernels,
    thousands of reads per grid"""
    rng = np.random.default_rng(505)
    reads = [synth.make_read(k, int(n), seed=505) for k, n in enumerate(rng.integers(500, 3001, 10500))]
    for k, n in enumerate((100_003, 256_000, 299_999, 170_000)):
        reads.insert(int(rng.integers(0, len(reads))), synth.make_read(20000 + k, n, seed=506))
    premise("reads over the warps of gen_prefix / gen_detect / gen_emit", len(reads), cap["gen_warp_reads"], 2.0)
    premise("reads over gen_tstat_kernel's CTAs", len(reads), cap["gen_tstat_reads"], 2.0)
    ctx = contexts.get(1 << 25, 16384, sg.F_FORCE_GENERIC)
    for rna in (0, 1):
        res = ctx.run(reads, rna=rna, want=sg.WANT_EVENTS)
        assert np.all(res.seq_order == 1)
        check_all(orc, res, reads, rna, sg.WANT_EVENTS)


def test_fast_and_sequential_order_reads_interleaved(contexts, orc, cap):
    """test 6: reads that fail the exact-sum witness next to reads on the fast path, and an 8-sample detector warm-up
    that sends more of them back: neighbouring reads share bitmap edge words, which clear_read_bits clears with
    atomicAnd while the fast path's bits of the read next door are already set"""
    rng = np.random.default_rng(606)
    lens = rng.integers(500, 9501, 12000)
    reads = [glitch_read(int(n), seed=6000 + k) if k % 2 else synth.make_read(k, int(n), seed=606)
             for k, n in enumerate(lens)]
    premise("verify_chunks_kernel items (128-sample chunks)", verify_items(lens, 128), cap["verify_chunks_items"], 1.3)
    ctx = contexts.get(1 << 26, 16384)
    with params(ctx, chunk_len=128, warmup=8):
        res = ctx.run(reads, rna=0, want=sg.WANT_EVENTS)
    n_seq = int(res.seq_order.sum())
    premise("sequential-order reads over the warps of gen_prefix / gen_detect / gen_emit", n_seq, cap["gen_warp_reads"])
    assert int(res.fixups.sum()) > 0
    assert np.all(res.seq_order[1::2] == 1) and np.all(res.seq_order[res.fixups > 0] == 1)
    check_all(orc, res, reads, 0, sg.WANT_EVENTS)


# ---- a context of production size: the sequential-order scratch is an eighth of it --------------------------------------
def test_scratch_of_an_eighth(contexts, orc, cap):
    """test 7: (a) reads that fail the witness, spread through a 70 M-sample batch and less than the scratch in all,
    are redone in order and are the only ones; (b) a batch whose fallback reads need more than the scratch is
    reported as SGPU_E_SCRATCH, not returned; (c) the next batch on the same context is exact again"""
    max_samples = 96 << 20
    gen_cap = max_samples // 8          # capi.cu:421 (contexts above 64 Mi samples without F_FULL_SEQ_SCRATCH)
    rng = np.random.default_rng(707)
    reads = synth.make_reads(1900, mean=36000.0, seed=707, hi=200000)
    glitch = np.zeros(len(reads) + 100, bool)
    glitch[np.sort(rng.choice(len(glitch), 100, replace=False))] = True
    it = iter(reads)
    reads = [glitch_read(30000, seed=7000 + k) if g else next(it) for k, g in enumerate(glitch)]
    premise("span (samples)", span_of(reads), 70e6)
    fallback = sum((len(rd[0]) + 7) // 8 * 8 for rd, g in zip(reads, glitch) if g)
    assert fallback < gen_cap, (fallback, gen_cap)
    ctx = contexts.get(max_samples, 4096)
    a = ctx.run(reads, rna=0, want=sg.WANT_EVENTS)
    assert np.array_equal(a.seq_order.astype(bool), glitch)
    check_all(orc, a, reads, 0, sg.WANT_EVENTS)
    with params(ctx, chunk_len=128, warmup=8):
        with pytest.raises(sg.SgpuError) as e:
            ctx.run(reads, rna=0, want=sg.WANT_EVENTS)
    assert e.value.code == -8          # SGPU_E_SCRATCH
    assert ctx.counters()["status"] == -8
    c = ctx.run(reads, rna=0, want=sg.WANT_EVENTS)
    assert ctx.counters()["status"] == 0
    assert np.array_equal(c.ev_off, a.ev_off) and np.array_equal(c.ev_start, a.ev_start)
    assert np.array_equal(bits(c.ev_mean), bits(a.ev_mean)) and np.array_equal(bits(c.ev_stdv), bits(a.ev_stdv))
    assert np.array_equal(c.seq_order, a.seq_order)


# ---- the long detector's job list ---------------------------------------------------------------------------------------
def check_thr_paths(orc, res, reads, rna, thr):
    """reads on the fast path use the lowered threshold of the long detector, the sequential-order kernels the
    reference's 9.0; -> number of event starts that only the lowered threshold gives"""
    def one(r):
        rd = reads[r]
        seq = bool(res.seq_order[r])
        st = orc.events(*rd, rna=rna)[0].astype(np.int64) if seq else event_starts_at(orc, rd, rna, thr)
        ok = np.array_equal(res.events(r).start.astype(np.int64), st)
        extra = 0 if seq else len(np.setdiff1d(st, orc.events(*rd, rna=rna)[0].astype(np.int64)))
        return r, seq, ok, extra
    out = pmap(one, range(len(reads)))
    bad = [(r, len(reads[r][0]), "sequential order" if seq else "fast path") for r, seq, ok, _ in out if not ok]
    assert not bad, f"{len(bad)} of {len(reads)} reads differ (read, length, path): {bad[:8]}"
    return sum(x for *_, x in out)


@pytest.mark.parametrize("rna", [0, 1])
def test_long_jobs_past_the_grid(contexts, orc, cap, rna):
    """test 8(a): with the long detector's threshold lowered it emits all the time; the replayed lives outnumber
    long_jobs_kernel's threads (DNA) or warps (RNA) several times over, and all fit in the job list"""
    thr = 0.3
    reads = synth.make_reads(800 if not rna else 400, mean=3000.0, seed=808 + rna, lo=500, hi=6000, rna=bool(rna))
    ctx = contexts.get(1 << 25, 8192)
    job_cap = (1 << 25) // 64 + 4096    # walk.cu:383
    with params(ctx, thr_long=thr):
        res = ctx.run(reads, rna=rna, want=sg.WANT_EVENTS)
        jobs = ctx.counters()["n_long_jobs"]
    print(f"rna={rna}: n_long_jobs {jobs} on {span_of(reads)} samples")
    premise("replayed lives over long_jobs_kernel's " + ("warps" if rna else "threads"), jobs,
            cap["long_jobs_rna" if rna else "long_jobs_dna"], 2.0)
    assert jobs < job_cap
    assert int(res.seq_order.sum()) == 0
    assert check_thr_paths(orc, res, reads, rna, thr) > 0


@pytest.mark.parametrize("rna", [0, 1])
def test_long_jobs_past_the_list(contexts, orc, rna):
    """test 8(b): a 2^20-sample context has room for 2^20 / 64 + 4,096 = 20,480 lives; a batch with more sends the
    reads whose lives did not fit to the sequential-order kernels (which keep the reference's threshold). Reads of a
    few dozen samples have a life or two each, so some of them keep all their lives in the list and stay on the fast
    path with the lowered threshold."""
    thr = 0.3
    max_samples = 1 << 20
    job_cap = max_samples // 64 + 4096
    rng = np.random.default_rng(818 + rna)
    reads, used = [], 0
    while True:
        n = int(rng.integers(500, 3001)) if len(reads) % 7 == 0 else int(rng.integers(16, 65))
        if used + (n + 7) // 8 * 8 > max_samples:
            break
        reads.append(synth.make_read(len(reads), n, seed=818 + rna))   # (DNA-like level changes: more lives for RNA)
        used += (n + 7) // 8 * 8
    ctx = contexts.get(max_samples, 4096)
    with params(ctx, thr_long=thr):
        res = ctx.run(reads, rna=rna, want=sg.WANT_EVENTS)
        jobs = ctx.counters()["n_long_jobs"]    # (the capped count: walk.cu:287-288)
    n_seq = int(res.seq_order.sum())
    print(f"rna={rna}: n_long_jobs {jobs} (capacity {job_cap}), {n_seq} of {len(reads)} reads in sequential order")
    assert jobs == job_cap
    assert 1 <= n_seq < len(reads)
    check_thr_paths(orc, res, reads, rna, thr)


# ---- a batch that fills its context exactly -------------------------------------------------------------------------------
def test_batch_fills_the_context(contexts, orc):
    """test 9: span == max_samples, the last read ending on the last sample: every bounds check at the end of the span
    meets the end of the allocation; through the host slots and through sgpu_run_device with a device tensor of exactly
    span samples"""
    torch = pytest.importorskip("torch")
    max_samples = 1 << 22
    rng = np.random.default_rng(909)
    reads, used = [], 0
    while max_samples - used > 60000:
        n = int(rng.integers(1, 30000))
        rd = adaptor_read(len(reads), n, seed=909) if len(reads) % 7 == 3 else synth.make_read(len(reads), n, seed=909)
        reads.append(rd)
        used += (n + 7) // 8 * 8
    reads.append(adaptor_read(len(reads), max_samples - used, seed=910))
    assert span_of(reads) == max_samples and len(reads[-1][0]) % 8 == 0
    ctx = contexts.get(max_samples, 1024)
    assert ctx.max_samples == max_samples
    for rna in (0, 1):
        res = ctx.run(reads, rna=rna, want=ALL6)
        check_all(orc, res, reads, rna, ALL6)
    # the same batch (RNA) from device memory
    lens = np.array([len(rd[0]) for rd in reads], np.int64)
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(max_samples, np.int16)
    for r, rd in enumerate(reads):
        flat[off[r]:off[r] + lens[r]] = rd[0]
    dev = torch.device("cuda:0")
    d_s = torch.from_numpy(flat).to(dev)
    assert d_s.numel() == max_samples
    d_off = torch.from_numpy(off).to(dev)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    d_o = torch.tensor([np.float32(rd[2]) for rd in reads], dtype=torch.float32, device=dev)
    d_u = torch.tensor([np.float32(np.float32(rd[3]) / np.float32(rd[1])) for rd in reads], dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    d = ctx.run_device(d_s.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_o.data_ptr(), d_u.data_ptr(), len(reads),
                       max_samples, 1, ALL6, st)
    torch.cuda.synchronize()
    c = ctx.counters()
    n, ne = len(reads), c["n_events"]
    assert c["status"] == 0 and ne == int(res.ev_off[-1])
    assert np.array_equal(ctx.d2h(d.ev_off, np.uint64, n + 1), res.ev_off)
    assert np.array_equal(ctx.d2h(d.ev_start, np.uint32, ne), res.ev_start)
    assert np.array_equal(bits(ctx.d2h(d.ev_mean, np.float32, ne)), bits(res.ev_mean))
    assert np.array_equal(bits(ctx.d2h(d.ev_stdv, np.float32, ne)), bits(res.ev_stdv))
    assert np.array_equal(bits(ctx.d2h(d.stat, np.float32, n * 6).reshape(n, 6)), bits(res.stat))
    assert np.array_equal(ctx.d2h(d.ent, np.float64, n * 3).reshape(n, 3), res.ent)
    assert np.array_equal(ctx.d2h(d.prefix_pos, np.int32, n * 4).reshape(n, 4), res.prefix_pos)
    assert np.array_equal(bits(ctx.d2h(d.prefix_stat, np.float32, n * 6).reshape(n, 6)), bits(res.prefix_stat))
    pa = ctx.d2h(d.pa, np.float32, max_samples)
    cnt = ctx.d2h(d.jnn_cnt, np.uint32, n)
    seg = ctx.d2h(d.jnn_seg, np.int32, 2 * ((max_samples >> 5) + n + 1)).reshape(-1, 2)
    for r in range(n):
        assert np.array_equal(bits(pa[off[r]:off[r] + lens[r]]), bits(res.pa[r])), f"read {r}: pA differs"
        base = (int(off[r]) >> 5) + r   # SGPU_JNN_BASE
        assert np.array_equal(seg[base:base + int(cnt[r])].astype(np.int64), res.jnn[r]), f"read {r}: jnn differs"


# ---- RNA004 pores -----------------------------------------------------------------------------------------------------------
def short_adaptor_read(k, seed=31):
    """an RNA-like read with a dip of 500-1,999 samples near its start and a high stretch (clamped to 1,200 by jnnv2)
    in its second half that widens the band: depending on the depth, the run below the band's lower edge is long enough
    for RNA004's shortest run (500) but not for R9's (2,000), or the lower edge of RNA004 (0.7 stdv) misses it"""
    rng = np.random.default_rng([seed, k])
    n = int(rng.integers(24000, 40000))
    rd = synth.make_read(k, n, seed=seed, p_change=0.025)
    raw = rd[0].astype(np.int32)
    d = int(rng.integers(500, 2000))
    a0 = int(rng.integers(500, 3000))
    raw[a0:a0 + d] -= int(round(rng.uniform(10.0, 40.0) * synth.DIGITISATION / synth.RANGE))
    h0 = int(rng.integers(n // 2, n - 2500))
    raw[h0:h0 + n // 20] = 1300
    return np.clip(raw, -32768, 32767).astype(np.int16), rd[1], rd[2], rd[3]


def test_prefix_rna004(contexts, orc):
    """SGPU_PARAM_PORE = 1 gives jnnv2 the parameters of JNNV2_RNA_RNA004_ADAPTOR (std_scale 0.7, shortest run 500,
    jnn.h:88-102): every read matches the oracle under both pores, and short adaptors that only RNA004 accepts are
    found under RNA004 and not under R9 -- the parameter reaches the kernel"""
    reads = [adaptor_read(k, int(n), seed=17) for k, n in enumerate([30000, 45000, 60000, 90000, 25000, 150000, 33333])]
    reads += [adaptor_read(50 + k, 40000, seed=18, polya=False) for k in range(3)]
    reads += [short_adaptor_read(k) for k in range(40)]
    ctx = contexts.get(1 << 22, 1024)
    got = {}
    for pore in (0, 1):
        with params(ctx, pore=pore):
            res = ctx.run(reads, rna=1, want=sg.WANT_PREFIX)
        check_all(orc, res, reads, 1, sg.WANT_PREFIX, pore=pore)
        got[pore] = res.prefix_pos
    only4 = int(((got[1][:, 1] > 0) & (got[0][:, 1] <= 0)).sum())
    only9 = int(((got[0][:, 1] > 0) & (got[1][:, 1] <= 0)).sum())
    print(f"adaptors found under RNA004 only: {only4}, under R9 only: {only9}")
    assert only4 >= 5
    assert int((got[1][:10, 1] > 0).sum()) >= 5       # the long adaptors of adaptor_read are found under RNA004 too

"""GPU tests of SGPU_WANT_JNN with the caller's own parameters (sgpu_set_jnn, Context.set_jnn): the reference's sets
given explicitly reproduce the default path and the reference's stdout; custom sets on both routes (the automaton of
jnn_walk_kernel for error <= 6 < corrector, jnn_exact_kernel for every other set) equal orc_jnn_set
(tests/tools/jnn_set_oracle.c) read by read; the other products of a batch do not change; a host slot keeps the set in
force at its submit; refused sets leave the previous one in place. Everything is compared exactly."""
import os

import numpy as np
import pytest

import _fmt
from _jnn_ref import JnnSetRef, random_set, stall_reads
from _oracle import Oracle
import sigtk_b200 as sg

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
E_INVAL = -1
ALL_WANTS = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX

# the automaton route: error <= 6 < corrector
AUTOMATON = {
    "custom": sg.Jnn(188, 0.25, 4, 60, 50, 0.7),
    "error6": sg.Jnn(300, 0.5, 6, 80, 7, 0.9),        # eight states: every 3-bit field of a map in use
    "error0": sg.Jnn(64, 0.5, 0, 20, 1, 1.0),         # two states
    "negative_merge": sg.Jnn(1200, 0.05, 3, -5, 9, 0.6),
}
# the exact route: error >= corrector (the corrector's decrement acts), or error > 6
EXACT = {
    "error_is_corrector": sg.Jnn(150, 0.25, 50, 50, 50, 0.75),
    "error40": sg.Jnn(188, 0.25, 40, 60, 10, 0.7),    # tails longer than a word
    "corrector0": sg.Jnn(64, 1.0, 2, 50, 0, 0.75),
    "error40_no_decrement": sg.Jnn(200, 0.5, 40, 50, 100, 0.75),
}


@pytest.fixture(scope="module")
def ref():
    return JnnSetRef()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=1 << 25, max_reads=8192) as c:
        yield c
        c.set_jnn(None)


@pytest.fixture(autouse=True)
def no_set_between_tests(ctx):
    ctx.set_jnn(None)
    yield
    ctx.set_jnn(None)


def edge_reads():
    """an empty read, a 1-sample read, a read clipped flat at 1200, and stretches of exactly 32 in-band samples"""
    flat32 = np.tile(np.r_[np.full(32, 500, np.int16), np.int16(900)], 100)
    return [(np.zeros(0, np.int16), 8192.0, 0.0, 1400.0), (np.array([700], np.int16), 8192.0, 0.0, 1400.0),
            (np.full(3000, 1300, np.int16), 8192.0, 0.0, 1400.0), (flat32, 8192.0, 0.0, 1400.0)]


def long_read(seed, n=2_000_000):
    """one read of n samples with stalls all along it"""
    rng = np.random.default_rng(seed)
    raw = (500 + 60 * rng.standard_normal(n)).astype(np.int64)
    pos = 0
    while pos < n:
        stop = min(n, pos + int(rng.integers(20, 3000)))
        raw[pos:stop] = 500 + rng.integers(-6, 7, stop - pos)
        if rng.integers(0, 2):
            raw[rng.integers(pos, stop, int(rng.integers(1, 50)))] = 900
        pos = stop + int(rng.integers(3, 2000))
    raw[::7919] = 9000
    return (np.clip(raw, -32768, 32767).astype(np.int16), 8192.0, 3.0, 1400.0)


def check(ref, res, reads, p, what):
    n_seg = 0
    for r, rd in enumerate(reads):
        exp = ref.jnn(rd[0], p)
        assert np.array_equal(res.jnn[r], exp), f"{what} {tuple(p)}: read {r} of {len(rd[0])}: {res.jnn[r][:4]} vs {exp[:4]}"
        n_seg += len(exp)
    return n_seg


def device_jnn(torch, c, reads, rna, want=sg.WANT_JNN):
    """sgpu_run_device on device copies of `reads`; -> per read int64[k][2] segments"""
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
    assert c.counters()["status"] == 0
    n = len(reads)
    cnt = c.d2h(d.jnn_cnt, np.uint32, n)
    seg = c.d2h(d.jnn_seg, np.int32, 2 * ((int(off[-1]) >> 5) + n + 1)).reshape(-1, 2)
    return [seg[(int(off[r]) >> 5) + r:][:int(cnt[r])].astype(np.int64) for r in range(n)]


def same_products(a, b):
    """the outputs other than JNN of two host results of the same batch, by their bits"""
    for x, y in ((a.ev_off, b.ev_off), (a.ev_start, b.ev_start), (a.ev_mean, b.ev_mean), (a.ev_stdv, b.ev_stdv),
                 (a.stat, b.stat), (a.ent, b.ent), (a.prefix_pos, b.prefix_pos), (a.prefix_stat, b.prefix_stat)):
        if x is None or y is None or not np.array_equal(np.ascontiguousarray(x).view(np.uint8),
                                                        np.ascontiguousarray(y).view(np.uint8)):
            return False
    return all(np.array_equal(p.view(np.uint32), q.view(np.uint32)) for p, q in zip(a.pa, b.pa))


# ---- the reference's sets given explicitly ---------------------------------------------------------------------------
@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_jnn", 0), ("synth_rna.npz", "ref_rna_jnn", 1),
                                              ("jnn_stalls_dna.npz", "ref_jnn_stalls_dna", 0),
                                              ("jnn_stalls_rna.npz", "ref_jnn_stalls_rna", 1)])
def test_explicit_reference_set_is_the_default(ctx, orc, npz, txt, rna_flag):
    torch = pytest.importorskip("torch")
    named = _fmt.load_npz(os.path.join(G, npz))
    reads = [rd for _, rd in named]
    svb = [(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads]
    runs = {}
    for name, p in (("default", None), ("explicit", sg.Jnn.DRNA_R9 if rna_flag else sg.Jnn.CDNA_R9)):
        ctx.set_jnn(p)
        runs[name] = (ctx.run(reads, rna=rna_flag, want=sg.WANT_JNN).jnn,
                      ctx.run_svbzd(svb, rna=rna_flag, want=sg.WANT_JNN).jnn, device_jnn(torch, ctx, reads, rna_flag))
        if p is not None:  # under the other rna too: rna no longer chooses the jnn parameters
            runs[name] += (ctx.run(reads, rna=1 - rna_flag, want=sg.WANT_JNN).jnn,)
    for k, what in enumerate(("int16", "svb-zd", "device", "other rna")):
        got = runs["explicit"][k]
        assert all(np.array_equal(got[r], runs["default"][0][r]) for r in range(len(reads))), what
    for compact, suffix in ((False, ".txt"), (True, "_c.txt")):
        text = _fmt.JNN_HDR + "".join(_fmt.jnn_line(rid, len(rd[0]), runs["explicit"][0][r], compact)
                                      for r, (rid, rd) in enumerate(named))
        assert text == open(os.path.join(G, txt + suffix)).read(), suffix


# ---- custom sets on both routes ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(AUTOMATON) + sorted(EXACT))
def test_custom_set_stall_batches_vs_oracle(ctx, ref, name):
    """hundreds of seeded stall reads with ragged lengths, outliers inside the stalls, clipped spikes, an empty and a
    1-sample read; the other products of the same batch bit for bit as without the set"""
    p = AUTOMATON.get(name) or EXACT[name]
    rng = np.random.default_rng(sorted(AUTOMATON).index(name) if name in AUTOMATON else 10 + sorted(EXACT).index(name))
    reads = stall_reads(rng, 300 if p.window < 500 else 120, p.window, outlier_every=2) + edge_reads()
    base = ctx.run(reads, rna=0, want=ALL_WANTS)
    ctx.set_jnn(p)
    res = ctx.run(reads, rna=0, want=ALL_WANTS)
    n_seg = check(ref, res, reads, p, name)
    assert n_seg > len(reads), n_seg
    assert same_products(res, base)
    if name in EXACT and p.error >= p.corrector:  # the corrector's decrement acts on these reads
        assert sum(ref.decrements(rd[0], p) for rd in reads) > 0


@pytest.mark.parametrize("p", [AUTOMATON["custom"], AUTOMATON["error6"], EXACT["error40"], EXACT["corrector0"]])
def test_custom_set_long_read_svbzd_and_device(ctx, orc, ref, p):
    """one read of 2,000,000 samples among short ones, as int16 records, svb-zd streams and device-resident"""
    torch = pytest.importorskip("torch")
    reads = [long_read(5)] + stall_reads(np.random.default_rng(6), 20, p.window) + edge_reads()
    ctx.set_jnn(p)
    res = ctx.run(reads, rna=1, want=sg.WANT_JNN)
    assert check(ref, res, reads, p, "int16") > 500
    sres = ctx.run_svbzd([(orc.svbzd_encode(rd[0]), rd[1], rd[2], rd[3]) for rd in reads], rna=1, want=sg.WANT_JNN)
    dres = device_jnn(torch, ctx, reads, 1)
    for r in range(len(reads)):
        assert np.array_equal(sres.jnn[r], res.jnn[r]), f"svb-zd read {r}"
        assert np.array_equal(dres[r], res.jnn[r]), f"device read {r}"


@pytest.mark.parametrize("route", ["automaton", "exact"])
def test_more_reads_than_one_wave(ctx, ref, route):
    """8,000 reads (more warps than the GPU holds at once), seeded sets of the route"""
    rng = np.random.default_rng(31 if route == "automaton" else 32)
    p = sg.Jnn(*random_set(rng, automaton=route == "automaton"))
    reads = []
    for k in range(8000):
        n = int(rng.integers(0, 3000))
        raw = (500 + 50 * rng.standard_normal(n)).astype(np.int64)
        a = int(rng.integers(0, max(n, 1)))
        stall = raw[a:a + 2 * p.window]
        stall[:] = 500 + rng.integers(-4, 5, len(stall))
        reads.append((raw.astype(np.int16), 8192.0, 0.0, 1400.0))
    ctx.set_jnn(p)
    res = ctx.run(reads, rna=0, want=sg.WANT_JNN)
    assert check(ref, res, reads, p, route) > 20


def test_smallest_set_fills_the_segment_slots(ctx, ref):
    """window 32, stall_len 1.0: stretches of 32 in-band samples closed by one outlier, n/33 segments per read against
    n/32 + 1 slots, reads back to back"""
    p = sg.Jnn(32, 1.0, 0, 0, 1, 0.75)
    unit = np.r_[np.full(32, 500, np.int16), np.int16(900)]
    reads = [(np.tile(unit, k), 8192.0, 0.0, 1400.0) for k in (1, 2, 31, 32, 33, 1000, 60000)]
    reads += [(np.r_[np.tile(unit, 50), np.full(7, 500, np.int16)], 8192.0, 0.0, 1400.0)]
    ctx.set_jnn(p)
    res = ctx.run(reads, rna=0, want=sg.WANT_JNN | sg.WANT_STAT)
    check(ref, res, reads, p, "smallest")
    assert len(res.jnn[6]) == 60000
    ctx.set_jnn(sg.Jnn(32, 1.0, 7, 0, 1, 0.75))  # the same on the exact route: error > 6
    check(ref, ctx.run(reads, rna=0, want=sg.WANT_JNN), reads, sg.Jnn(32, 1.0, 7, 0, 1, 0.75), "smallest exact")


# ---- when the set takes effect -------------------------------------------------------------------------------------
def test_slot_keeps_the_set_of_its_submit(ctx, ref, orc):
    a, b = AUTOMATON["custom"], EXACT["error40"]
    reads = stall_reads(np.random.default_rng(12), 60, 188, outlier_every=1)
    ctx.set_jnn(a)
    ctx.fill(0, reads, 0)
    ctx.submit(0, sg.WANT_JNN)
    ctx.set_jnn(b)
    ctx.fill(1, reads, 0)
    ctx.submit(1, sg.WANT_JNN)
    ctx.set_jnn(None)
    r0, r1 = ctx.wait(0, sg.WANT_JNN), ctx.wait(1, sg.WANT_JNN)
    check(ref, r0, reads, a, "slot 0")
    check(ref, r1, reads, b, "slot 1")
    assert any(not np.array_equal(r0.jnn[r], r1.jnn[r]) for r in range(len(reads)))
    res = ctx.run(reads, rna=0, want=sg.WANT_JNN)
    for r, rd in enumerate(reads):
        assert np.array_equal(res.jnn[r], orc.jnn(rd[0], 0)), f"after set_jnn(None): read {r}"


# ---- refusals ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [
    sg.Jnn(150, 0.25, -1, 50, 50, 0.75),             # error < 0
    sg.Jnn(150, 0.25, 5, 50, -1, 0.75),              # corrector < 0
    sg.Jnn(150, float("nan"), 5, 50, 50, 0.75),      # stall_len not finite
    sg.Jnn(150, float("inf"), 5, 50, 50, 0.75),
    sg.Jnn(150, 0.25, 5, 50, 50, float("nan")),      # std_scale not finite
    sg.Jnn(150, 0.25, 5, 50, 50, float("-inf")),
    sg.Jnn(31, 2.0, 5, 50, 50, 0.75),                # window <= 31
    sg.Jnn(0, 100.0, 5, 50, 50, 0.75),
    sg.Jnn(-150, -0.25, 5, 50, 50, 0.75),
    sg.Jnn(62, 0.5, 5, 50, 50, 0.75),                # window * stall_len = 31
    sg.Jnn(100, 0.3, 5, 50, 50, 0.75),               # fl(100 * 0.3f) = 30.000002
    sg.Jnn(150, -0.25, 5, 50, 50, 0.75),
])
def test_refused_set_keeps_the_previous(ctx, ref, bad):
    keep = EXACT["corrector0"]
    ctx.set_jnn(keep)
    with pytest.raises(sg.SgpuError) as e:
        ctx.set_jnn(bad)
    assert e.value.code == E_INVAL
    reads = stall_reads(np.random.default_rng(3), 20, 64, outlier_every=1)
    check(ref, ctx.run(reads, rna=0, want=sg.WANT_JNN), reads, keep, "after a refusal")


def test_boundary_sets_are_accepted(ctx, ref):
    reads = stall_reads(np.random.default_rng(4), 10, 64)
    for p in (sg.Jnn(32, 1.0, 5, 50, 50, 0.75), sg.Jnn(63, 0.5, 5, 50, 50, 0.75), sg.Jnn(40, 1.0, 0, 0, 0, -0.5)):
        ctx.set_jnn(p)
        check(ref, ctx.run(reads, rna=0, want=sg.WANT_JNN), reads, p, "boundary")

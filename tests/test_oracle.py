"""Pins the CPU oracle (oracle/sigtk_oracle.c) to the reference:
   - the reference's own golden file test/event_dna.exp (scripts/test.sh:70-72),
   - stdout of the compiled, unmodified reference (fixtures in tests/golden/, made by make_golden.py),
   - stdout of the compiled reference and the svb-zd streams of its slow5lib on seeded synthetic reads
     (sha256 in tests/golden/ref_outputs.json, made by make_ref_outputs.py).
CPU only."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

import _fmt
import _refcases
from _oracle import Oracle
from sigtk_b200 import synth

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_OUT = json.load(open(os.path.join(G, "ref_outputs.json")))


def _sha(b):
    return hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


@pytest.fixture(scope="module")
def sp1():
    return _fmt.load_npz(os.path.join(G, "sp1_dna.npz"))


@pytest.fixture(scope="module")
def rna():
    return _fmt.load_npz(os.path.join(G, "synth_rna.npz"))


def test_event_dna_exp(orc, sp1):
    """the reference's own golden: long-form events of read 05d90f17-... (header line of the .exp is stale)"""
    exp = open(os.path.join(G, "event_dna.exp")).read().split("\n", 1)[1]
    rid, rd = next(x for x in sp1 if x[0] == "05d90f17-f4a6-4349-924c-3ffd3457a99d")
    got = _fmt.event_long(rid, *orc.events(*rd))
    assert got == exp
    assert got.count("\n") == 915 + 1


def test_sp1_event_compact_all_reads(orc, sp1):
    exp = open(os.path.join(G, "ref_sp1_event_c.txt")).read()
    got = _fmt.EVENT_HDR_COMPACT
    total = 0
    for rid, rd in sp1:
        st, ln, _, _ = orc.events(*rd)
        total += len(st)
        got += _fmt.event_compact(rid, len(rd[0]), st, ln)
    assert got == exp
    assert total == 92935  # SURVEY 8(a) C1


def test_sp1_event_long_first10(orc, sp1):
    exp = gzip.open(os.path.join(G, "ref_sp1_event_first10.txt.gz"), "rt").read()
    got = _fmt.EVENT_HDR_LONG + "".join(_fmt.event_long(rid, *orc.events(*rd)) for rid, rd in sp1[:10])
    assert got == exp


def test_sp1_pa_first10(orc, sp1):
    exp = gzip.open(os.path.join(G, "ref_sp1_pa_first10.txt.gz"), "rt").read()
    got = _fmt.PA_HDR + "".join(_fmt.pa_line(rid, orc.pa(*rd)) for rid, rd in sp1[:10])
    assert got == exp


def test_sp1_stat(orc, sp1):
    exp = open(os.path.join(G, "ref_sp1_stat.txt")).read()
    got = _fmt.STAT_HDR + "".join(_fmt.stat_line(rid, len(rd[0]), orc.stat(*rd)) for rid, rd in sp1)
    assert got == exp


def test_rna_event_long_and_compact(orc, rna):
    exp = gzip.open(os.path.join(G, "ref_rna_event.txt.gz"), "rt").read()
    got = _fmt.EVENT_HDR_LONG + "".join(_fmt.event_long(rid, *orc.events(*rd, rna=1)) for rid, rd in rna)
    assert got == exp
    exp = open(os.path.join(G, "ref_rna_event_c.txt")).read()
    got = _fmt.EVENT_HDR_COMPACT
    for rid, rd in rna:
        st, ln, _, _ = orc.events(*rd, rna=1)
        got += _fmt.event_compact(rid, len(rd[0]), st, ln)
    assert got == exp


def test_rna_stat(orc, rna):
    exp = open(os.path.join(G, "ref_rna_stat.txt")).read()
    got = _fmt.STAT_HDR + "".join(_fmt.stat_line(rid, len(rd[0]), orc.stat(*rd)) for rid, rd in rna)
    assert got == exp


# ---- `sigtk ent` (SURVEY 8f rank 4) ---------------------------------------------------------------
@pytest.mark.parametrize("npz,txt", [("sp1_dna.npz", "ref_sp1_ent.txt"), ("synth_rna.npz", "ref_rna_ent.txt"),
                                     ("ent_adversarial.npz", "ref_ent_adversarial.txt")])
def test_ent_equals_reference_stdout(orc, npz, txt):
    """orc_ent against the stdout of the compiled reference's `sigtk ent` (same libm: bit-identical doubles, so the
    text must be identical), including reads with wrapped / wide / single-bin histograms and 1- and 2-sample records"""
    reads = _fmt.load_npz(os.path.join(G, npz))
    exp = open(os.path.join(G, txt)).read()
    got = _fmt.ENT_HDR + "".join(_fmt.ent_line(rid, orc.ent(rd[0])) for rid, rd in reads)
    assert got == exp


def test_ent_against_numpy_histograms(orc):
    """independent restatement with numpy (bincount + log2; pairwise instead of sequential summation, hence 1e-10);
    also where the reference aborts (|delta| >= 16384)"""
    rng = np.random.default_rng(5)
    for raw in (rng.integers(-32768, 32768, 50000).astype(np.int16), rng.integers(300, 900, 777).astype(np.int16),
                np.array([7], dtype=np.int16), np.zeros(0, dtype=np.int16)):
        def H(keys, total):
            c = np.bincount(keys, minlength=1)
            p = c[c > 0] / float(total)
            return float(-(p * np.log2(p)).sum()) if total else 0.0
        n = raw.shape[0]
        exp = np.zeros(3)
        if n:
            exp[0] = H(raw.view(np.uint16).astype(np.int64), n)
        if n > 1:
            d = np.diff(np.concatenate([[0], raw.astype(np.int64)]))[: n - 1]
            z = (((d << 1) ^ (d >> 63)) & 0xffff)
            exp[1] = H(z, n - 1)
            exp[2] = H(z >> 8, n - 1) + H(z & 255, n - 1)
        assert np.allclose(orc.ent(raw), exp, rtol=0, atol=1e-10)


# ---- `sigtk jnn` (SURVEY 8f rank 3, the jnn half) ----------------------------------------------------
@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_jnn", 0), ("synth_rna.npz", "ref_rna_jnn", 1),
                                              ("jnn_stalls_dna.npz", "ref_jnn_stalls_dna", 0),
                                              ("jnn_stalls_rna.npz", "ref_jnn_stalls_rna", 1)])
def test_jnn_equals_reference_stdout(orc, npz, txt, rna_flag):
    """orc_jnn against the stdout of the compiled reference's `sigtk jnn` and `jnn -c`: real DNA, synthetic RNA, and
    reads with stalls (merged pairs, tolerated outliers, open stretches at the end, clipped spikes, empty band)"""
    reads = _fmt.load_npz(os.path.join(G, npz))
    for compact, suffix in ((False, ".txt"), (True, "_c.txt")):
        exp = open(os.path.join(G, txt + suffix)).read()
        got = _fmt.JNN_HDR + "".join(_fmt.jnn_line(rid, len(rd[0]), orc.jnn(rd[0], rna_flag), compact) for rid, rd in reads)
        assert got == exp, suffix


# ---- `sigtk prefix` (SURVEY 8f rank 3, prefix half): oracle only, the CUDA path is next round's --------------------
@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_prefix_stat.txt", 0),
                                              ("synth_rna.npz", "ref_rna_prefix_stat.txt", 1),
                                              ("prefix_adaptor_dna.npz", "ref_prefix_adaptor_dna_stat.txt", 0),
                                              ("prefix_adaptor_rna.npz", "ref_prefix_adaptor_rna_stat.txt", 1)])
def test_prefix_equals_reference_stdout(orc, npz, txt, rna_flag):
    """orc_adaptor_polya against `sigtk prefix --print-stat` (and, without the statistics, `sigtk prefix`) of the
    compiled reference: adaptor by jnnv2 on the rolling mean, poly-A by jnn_core on pA, float statistics of both"""
    reads = _fmt.load_npz(os.path.join(G, npz))
    rows = [(rid, len(rd[0])) + orc.adaptor_polya(*rd, rna=rna_flag) for rid, rd in reads]
    got = _fmt.PREFIX_HDR + _fmt.PREFIX_HDR_STAT + "\n" + "".join(_fmt.prefix_line(r, n, p, s, True) for r, n, p, s in rows)
    assert got == open(os.path.join(G, txt)).read()
    plain = txt.replace("_stat.txt", ".txt")
    if os.path.exists(os.path.join(G, plain)):
        got = _fmt.PREFIX_HDR + "\n" + "".join(_fmt.prefix_line(r, n, p, s, False) for r, n, p, s in rows)
        assert got == open(os.path.join(G, plain)).read()


def test_prefix_dna_exp(orc, sp1):
    """the reference's own golden test/prefix_dna.exp (scripts/test.sh:54-56)"""
    got = _fmt.PREFIX_HDR + "\n" + "".join(_fmt.prefix_line(rid, len(rd[0]), *orc.adaptor_polya(*rd, rna=0))
                                           for rid, rd in sp1)
    assert got == open(os.path.join(G, "prefix_dna.exp")).read()


@pytest.mark.parametrize("rna_flag,seed", _refcases.ORACLE_CASES)
def test_oracle_equals_compiled_reference(orc, rna_flag, seed):
    """the oracle's events, pA and stat of seeded synthetic reads, printed as the reference prints them, equal the
    stdout of the compiled reference's `sigtk event`, `pa` and `stat` on a BLOW5 of the same reads"""
    out = {"event": [_fmt.EVENT_HDR_LONG], "pa": [_fmt.PA_HDR], "stat": [_fmt.STAT_HDR]}
    for rid, *rd in _refcases.oracle_reads(rna_flag, seed):
        out["event"].append(_fmt.event_long(rid, *orc.events(*rd, rna=rna_flag)))
        out["pa"].append(_fmt.pa_line(rid, orc.pa(*rd)))
        out["stat"].append(_fmt.stat_line(rid, len(rd[0]), orc.stat(*rd)))
    want = REF_OUT["oracle"][f"{rna_flag}-{seed}"]
    for mode, parts in out.items():
        assert _sha("".join(parts).encode()) == want[mode], mode


def test_stagewise_consistency(orc):
    """the staged entry points compose to the same events as the one-shot call"""
    rd = synth.make_read(3, 12000)
    pa = orc.pa(*rd)
    S, Q = orc.prefix(pa)
    p = orc.params(0)
    t1, t2 = orc.tstat(S, Q, p.w_short), orc.tstat(S, Q, p.w_long)
    peaks, _, _ = orc.detect(t1, t2, 0)
    st, _, _, _ = orc.events(*rd)
    assert np.array_equal(np.concatenate([[0], peaks]).astype(np.uint64), st)
    assert np.all(np.diff(peaks.astype(np.int64)) >= 3)  # min peak gap floor(w1/2)+2 (SURVEY 7.3(4))


def test_detector_cold_start_adversarial(orc):
    """SURVEY 7.3(2): a sub-threshold peak held across a flat stretch makes cold-start states differ forever
    while the emitted peaks agree."""
    n = 1200
    t1 = np.zeros(n, dtype=np.float32)
    t1[10], t1[900] = 0.5, 3.0
    t2 = np.zeros(n, dtype=np.float32)
    peaks_true, s_true, _ = orc.detect(t1, t2, 0, 0, 500)
    peaks_cold, s_cold, _ = orc.detect(t1, t2, 0, 400, 500, cold=True)
    assert s_true[1:3] == (10, 0.5) and s_cold[1] == -1
    full, _, _ = orc.detect(t1, t2, 0)
    assert list(full) == [900]


def test_degenerate_inputs_defined(orc):
    """where the reference aborts (n<200, constant signal, zero peaks) the oracle defines one event [0,n)"""
    raw = np.full(50, 500, dtype=np.int16)
    st, ln, mn, sd = orc.events(raw, 8192.0, 10.0, 1400.0)
    assert list(st) == [0] and list(ln) == [50.0]
    st, ln, _, _ = orc.events(np.array([7], dtype=np.int16), 8192.0, 10.0, 1400.0)
    assert list(st) == [0] and list(ln) == [1.0]


# ---- svb-zd signal streams (SURVEY 8f rank 1; slow5_press.c:1055-1150) ----------------------------------------------
@pytest.fixture(scope="module")
def svb_golden():
    d = np.load(os.path.join(G, "svbzd_golden.npz"))
    return {k[4:]: (d["raw_" + k[4:]], d["svb_" + k[4:]]) for k in d.files if k.startswith("raw_")}


def test_svbzd_golden_streams(orc, svb_golden):
    """streams written by the reference's slow5lib (tests/golden/make_svbzd_golden.py): our decode gives the raw
    signal, our encode gives the same bytes (the encoder never emits 4-byte values for int16 input, so the
    hand-made wide-code stream is decode-only)"""
    assert len(svb_golden) >= 10
    for name, (raw, st) in svb_golden.items():
        dec = orc.svbzd_decode(st)
        assert dec is not None and np.array_equal(dec, raw), name
        if name != "wide_codes":
            assert np.array_equal(orc.svbzd_encode(raw), st), name


def test_svbzd_malformed_rejected(orc, svb_golden):
    raw, st = svb_golden["walk"]
    assert orc.svbzd_decode(st[:-1], cap=len(raw)) is None      # truncated data
    assert orc.svbzd_decode(np.concatenate([st, st[-1:]]), cap=len(raw)) is None  # trailing byte
    assert orc.svbzd_decode(st[:3]) is None                       # no header


def test_svbzd_equals_compiled_reference(orc):
    """the oracle's svb-zd encoder writes the bytes the reference's slow5lib stores (sha256 of each stream), and
    decodes them back"""
    raws = _refcases.svbzd_grid()
    assert len(raws) == len(REF_OUT["svbzd_grid"])
    for raw, want in zip(raws, REF_OUT["svbzd_grid"]):
        a = orc.svbzd_encode(raw)
        assert _sha(a.tobytes()) == want, len(raw)
        assert np.array_equal(orc.svbzd_decode(a), raw)


def test_synthetic_svbzd_encoder_equals_oracle(orc):
    """sigtk_b200.synth.svbzd_encode (numpy; makes compressed input for bench.py) writes the reference's bytes"""
    rng = np.random.default_rng(11)
    for n in (0, 1, 3, 4, 5, 1027, 20000):
        for scale in (5, 300, 50000):
            raw = np.clip(np.cumsum(rng.integers(-scale, scale + 1, n)), -32768, 32767).astype(np.int16)
            assert np.array_equal(synth.svbzd_encode(raw), orc.svbzd_encode(raw)), (n, scale)


def test_long_filter_checker_finds_no_violation(tmp_path):
    """oracle/proofs/long_filter_check.cpp: the float test that replaces the long window's t-statistic on the fast
    path (walk_core.cuh: long_candidate) never misses a position whose reference t2 exceeds the threshold
    (2,000,000 random / adversarial windows here; 10^9 in profiles/r02_long_filter_check.json)"""
    import subprocess
    exe = str(tmp_path / "long_filter_check")
    here = os.path.dirname(os.path.abspath(__file__))
    proofs = os.path.join(os.path.dirname(here), "oracle", "proofs")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-x", "c++",
                           os.path.join(proofs, "long_filter_check.cpp"), "-x", "c",
                           os.path.join(proofs, "..", "sigtk_oracle.c"), "-lm", "-o", exe], stderr=subprocess.DEVNULL)
    out = subprocess.run([exe, "2000000", "7"], check=True, stdout=subprocess.PIPE).stdout
    import json
    d = json.loads(out)
    assert d["violations"] == 0 and d["t_above_threshold"] > 500000


def test_window_division_shortcut_is_exact(tmp_path):
    """oracle/proofs/div_window_check.c: `sigtk prefix` divides the rolling-window sum by 2000 for every position; the
    CUDA path uses the reciprocal with one residual correction, which must equal the IEEE quotient for every value the
    (exact integer) sum can take -- checked for every integer up to 2^24."""
    import json
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    src = os.path.join(os.path.dirname(here), "oracle", "proofs", "div_window_check.c")
    exe = str(tmp_path / "div_window_check")
    subprocess.check_call(["gcc", "-O2", "-mfma", "-ffp-contract=off", src, "-o", exe, "-lm"])
    out = json.loads(subprocess.check_output([exe]).decode())
    assert out["mismatches"] == 0 and out["values"] == (1 << 24) + 1

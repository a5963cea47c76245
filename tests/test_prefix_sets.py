"""CPU tests of the restatement behind sgpu_set_prefix: tests/tools/prefix_set_oracle.c (prefix_func with every field
of the adaptor and poly-A sets general) equals the compiled reference's stored stdout and orc_adaptor_polya_pore with
the reference's sets; the poly-A corrector never acts on sets with error < corrector, and does act, changing the
result, on the exact-route sets the GPU tests use."""
import os

import numpy as np
import pytest

import _fmt
from _oracle import Oracle
from _prefix_ref import (ADAPTORS, AUTOMATON, POLYA_R9, REFERENCE, RNA_R9, PrefixSetRef, named_set,
                         random_set, set_read, without_corrector)
import sigtk_b200 as sg

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref():
    return PrefixSetRef()


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def test_python_sets_are_the_reference_sets():
    assert tuple(sg.Adaptor.RNA_R9) == REFERENCE[0][0] and tuple(sg.Adaptor.RNA004) == REFERENCE[1][0]
    assert tuple(sg.Polya.R9) == POLYA_R9
    assert tuple(sg.Prefix(sg.Adaptor.RNA_R9, sg.Polya.R9)) == REFERENCE[0]


@pytest.mark.parametrize("npz,txt,rna_flag", [("sp1_dna.npz", "ref_sp1_prefix_stat.txt", 0),
                                              ("synth_rna.npz", "ref_rna_prefix_stat.txt", 1),
                                              ("prefix_adaptor_dna.npz", "ref_prefix_adaptor_dna_stat.txt", 0),
                                              ("prefix_adaptor_rna.npz", "ref_prefix_adaptor_rna_stat.txt", 1)])
def test_reference_sets_equal_reference_stdout(ref, npz, txt, rna_flag):
    """`sigtk prefix --print-stat` and `sigtk prefix` of the compiled reference (R9 pore) from the restatement"""
    reads = _fmt.load_npz(os.path.join(G, npz))
    rows = [(rid, len(rd[0])) + ref.prefix(*rd, rna_flag, REFERENCE[0]) for rid, rd in reads]
    got = _fmt.PREFIX_HDR + _fmt.PREFIX_HDR_STAT + "\n" + "".join(_fmt.prefix_line(r, n, p, s, True) for r, n, p, s in rows)
    assert got == open(os.path.join(G, txt)).read()
    plain = txt.replace("_stat.txt", ".txt")
    if os.path.exists(os.path.join(G, plain)):
        got = _fmt.PREFIX_HDR + "\n" + "".join(_fmt.prefix_line(r, n, p, s, False) for r, n, p, s in rows)
        assert got == open(os.path.join(G, plain)).read()


def test_reference_sets_equal_prefix_dna_exp(ref):
    """the reference's own golden test/prefix_dna.exp"""
    reads = _fmt.load_npz(os.path.join(G, "sp1_dna.npz"))
    got = _fmt.PREFIX_HDR + "\n" + "".join(_fmt.prefix_line(rid, len(rd[0]), *ref.prefix(*rd, 0, REFERENCE[0]))
                                           for rid, rd in reads)
    assert got == open(os.path.join(G, "prefix_dna.exp")).read()


@pytest.mark.parametrize("pore", [0, 1])
@pytest.mark.parametrize("rna_flag", [0, 1])
def test_reference_sets_equal_oracle(ref, orc, pore, rna_flag):
    """both pores' sets against orc_adaptor_polya_pore on seeded reads (adaptors and poly-A tails of random length,
    reads around the window length, reads without an adaptor), positions and statistics bit for bit"""
    p = REFERENCE[pore]
    reads = [set_read(k, 40 + pore, p) for k in range(40)] + [set_read(k, 50, p, polya=False) for k in range(5)]
    base = set_read(99, 51, p)
    reads += [(base[0][:n].copy(),) + base[1:] for n in (1, 1999, 2000, 2001, 2002, 4001)]
    found = 0
    for rd in reads:
        pos, st = ref.prefix(*rd, rna_flag, p)
        opos, ost = orc.adaptor_polya(*rd, rna=rna_flag, pore=pore)
        assert np.array_equal(pos, opos)
        assert np.array_equal(bits(st), bits(ost))
        found += pos[1] > 0 and (pos[3] > 0 or not rna_flag)
    assert found >= 30


@pytest.mark.parametrize("seed", range(6))
def test_no_decrement_when_error_below_corrector(ref, seed):
    """the automaton route's premise: with error < corrector the poly-A corrector never decrements err"""
    rng = np.random.default_rng(700 + seed)
    n_found = 0
    for k in range(12):
        p = random_set(rng, exact=False)
        for q in (p, (RNA_R9, p[1])):   # the seeded adaptor set, and the R9 one
            pos, _, n_dec = ref._run(*set_read(k, 800 + seed, q), 1, q)
            assert n_dec == 0, q
            n_found += pos[3] > 0
    assert n_found > 0


@pytest.mark.parametrize("name", sorted(AUTOMATON) + sorted(ADAPTORS))
def test_named_automaton_sets_never_decrement(ref, name):
    p = named_set(name)
    assert all(ref.decrements(*set_read(k, 61, p), 1, p) == 0 for k in range(20))


@pytest.mark.parametrize("name", ["corrector0", "error_is_corrector", "error_above"])
def test_exact_sets_decrement_and_change_the_result(ref, name):
    """the exact-route sets of the GPU tests: the corrector fires on their reads, and a build that never stepped it
    would give other poly-A positions"""
    p = named_set(name)
    reads = [set_read(k, 71, p) for k in range(30)]
    assert sum(ref.decrements(*rd, 1, p) for rd in reads) > 0
    assert any(not np.array_equal(ref.prefix(*rd, 1, p)[0], ref.prefix(*rd, 1, without_corrector(p))[0])
               for rd in reads)


def test_error_max_decrements_without_overflow(ref):
    """error = INT32_MAX: every outlier is tolerated, a stretch never closes, no poly-A is found"""
    p = named_set("error_max")
    reads = [set_read(k, 72, p) for k in range(10)]
    assert sum(ref.decrements(*rd, 1, p) for rd in reads) > 0
    assert all(ref.prefix(*rd, 1, p)[0][3] == -1 for rd in reads)

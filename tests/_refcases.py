"""Inputs of the comparisons with the compiled, unmodified reference whose outputs are stored in
tests/golden/ref_outputs.json (made by tests/golden/make_ref_outputs.py). The tests and the generator build the same
inputs from these functions, so the stored outputs stay those of the inputs the tests use."""
from __future__ import annotations

import numpy as np

from sigtk_b200 import synth

ORACLE_CASES = [(0, 1), (0, 2), (1, 3)]  # (rna_flag, seed)
FUZZ_KINDS = ["genomic_dna", "rna"]


def oracle_reads(rna_flag: int, seed: int):
    """(read_id, raw, digitisation, offset, range) of 8 synthetic reads"""
    return [(f"synth-{seed}-{k}", *rd) for k, rd in
            enumerate(synth.make_reads(8, mean=15000.0, seed=seed, rna=bool(rna_flag)))]


def fuzz_reads(kind: str):
    """150 reads with glitches (pA <= 0), flat stretches, ramps, steps and saturation. Reads on which the reference
    aborts are left out: fewer than 1000 samples, and (its dead trimming step asserts on chunk-wise constant signals,
    events.c:242) reads whose first or last 200 samples do not vary."""
    from test_gpu_parity import _fuzz_read
    rng = np.random.default_rng(11 if kind == "rna" else 7)
    out, k = [], 0
    while len(out) < 150:
        raw, dig, off, rg = _fuzz_read(rng, k)
        k += 1
        if len(raw) < 1000 or np.ptp(raw[:200]) < 20 or np.ptp(raw[-200:]) < 20:
            continue
        out.append((f"fuzz-{k:05d}", raw, dig, off, rg))
    return out


def svbzd_grid():
    """int16 random walks: lengths around the key-byte and block sizes, 1-, 2- and 3-byte deltas"""
    rng = np.random.default_rng(5)
    raws = []
    for n in (0, 1, 2, 3, 4, 5, 31, 32, 33, 1023, 1024, 1025, 4097, 50001):
        for scale in (3, 200, 40000):
            raws.append(np.clip(np.cumsum(rng.integers(-scale, scale + 1, n)), -32768, 32767).astype(np.int16))
    return raws


def svbzd_reads():
    """24 synthetic reads (mean 30,000 samples)"""
    return [rd[0] for rd in synth.make_reads(24, mean=30000.0, seed=91)]

"""The contract of live event detection on the CPU: the streaming reference (tests/_live_ref.py) reports, over all the
chunks of a read, exactly the reference's event table of the whole read, for any split; and the ctypes mirror of the
live part of the C-ABI follows include/sigtk_b200.h."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from _live_ref import concat, same_events, split_lengths, stream_reference, whole_read
from _oracle import Oracle
from _oracle_pa import getevents_pa
from sigtk_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def golden(name):
    d = np.load(os.path.join(G, name))
    o = d["read_off"]
    return [(d["samples"][int(o[r]):int(o[r + 1])], float(d["digitisation"][r]), float(d["offset"][r]),
             float(d["range"][r])) for r in range(len(o) - 1)]


def sources():
    cb = [synth.make_read_cb(k, n) for k, n in enumerate((0, 1, 5, 13, 27, 28, 29, 600, 7000, 20000))]
    return [("cb_dna", cb, 0), ("cb_rna", cb, 1), ("sp1_dna", golden("sp1_dna.npz")[:30], 0),
            ("synth_rna", golden("synth_rna.npz")[:4], 1)]


@pytest.mark.parametrize("thr_long", [None, 1.0])
@pytest.mark.parametrize("src", range(4))
def test_concatenation_is_the_whole_read(orc, src, thr_long):
    name, reads, rna = sources()[src]
    rng = np.random.default_rng(1000 + src)
    for r, rd in enumerate(reads):
        pa = orc.pa(*rd)
        want = whole_read(orc, pa, rna, thr_long)
        if thr_long is None and len(pa):
            assert same_events(want, getevents_pa(orc, pa, rna)), f"{name} read {r}: whole-read reference"
        for _ in range(2):
            chunks = split_lengths(len(pa), rng)
            got, _ = stream_reference(orc, pa, rna, chunks, thr_long)
            assert len(got) == len(chunks)
            assert same_events(concat(got), want), f"{name} read {r} split {chunks[:8]}"


def long_read():
    """a read with a flat stretch and a slow ramp: lives of the long detector far from any short peak"""
    rd = synth.make_read(11, 30000, seed=3)
    raw = rd[0].copy()
    raw[6000:14000] = raw[5999]
    raw[14000:20000] = raw[5999] + (np.arange(6000) // 40)
    return (raw,) + rd[1:]


def late_long_peaks(orc, pa, rna, chunks, thr_long):
    """peaks that the lowered long threshold adds and that were emitted in a later chunk than the one in which their
    position was stepped"""
    peaks = stream_reference(orc, pa, rna, chunks, thr_long)[1]
    default = {q for q, _ in stream_reference(orc, pa, rna, chunks)[1]}
    stepped_by = np.cumsum(chunks) - orc.params(rna).w_long + 1
    return [q for q, k in peaks if q not in default and k > 0 and q < stepped_by[k - 1]]


@pytest.mark.parametrize("rna", [0, 1])
def test_long_detector_lives_span_chunks(orc, rna):
    """with the long threshold lowered, peaks of the long detector are emitted in a later chunk than the one in which
    their position was stepped, and the concatenation still is the whole read"""
    pa = orc.pa(*long_read())
    chunks = [37] * (len(pa) // 37) + [len(pa) % 37]
    got, _ = stream_reference(orc, pa, rna, chunks, thr_long=1.0)
    assert same_events(concat(got), whole_read(orc, pa, rna, 1.0))
    assert late_long_peaks(orc, pa, rna, chunks, 1.0), "no long-detector peak outlived its chunk"


def test_python_mirror_matches_the_header():
    hdr = open(os.path.join(ROOT, "include", "sigtk_b200.h")).read()
    defs = {k: int(v.rstrip("u"), 0) for k, v in re.findall(r"#define\s+(SGPU_[A-Z_]+)\s+(-?\d+u?)\b", hdr)}
    for name in ("START", "END", "RNA"):
        assert getattr(_lib, "LIVE_" + name) == defs["SGPU_LIVE_" + name]
    body = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for struct, mirror in (("sgpu_live_result_t", _lib.LiveResult), ("sgpu_dev_live_batch_t", _lib.DevLiveBatch)):
        decl = re.search(r"typedef struct \{([^}]*)\} " + struct + ";", body).group(1)
        names = []
        for line in filter(None, (x.strip() for x in decl.split(";"))):
            parts = line.split(",")
            names += [parts[0].split()[-1].lstrip("*")] + [x.strip().lstrip("*").strip() for x in parts[1:]]
        assert names == [f[0] for f in mirror._fields_], struct
    for fn in ("sgpu_live_open", "sgpu_slot_add_live", "sgpu_wait_live", "sgpu_run_device_live"):
        assert fn in _lib.EXPORTS


def test_null_context_is_refused():
    lib = _lib.load()
    raw = np.zeros(4, np.int16)
    assert lib.sgpu_live_open(None, 16) == -1
    assert lib.sgpu_slot_add_live(None, 0, 0, 1, raw.ctypes.data, 4, 8192.0, 0.0, 1400.0) == -1
    assert lib.sgpu_wait_live(None, 0, C.byref(_lib.LiveResult())) == -1
    assert lib.sgpu_run_device_live(None, C.byref(_lib.DevLiveBatch()), None, C.byref(_lib.LiveResult())) == -1

#!/usr/bin/env python
"""Generates tests/golden/ref_outputs.json and ref_fuzz_*.txt with the compiled, unmodified reference in oracle/_ref
(`make -C oracle ref`): the reference CLI `sigtk` and blow5_write / blow5_dump, which link the reference's slow5lib.

  oracle   sha256 of the stdout of `sigtk event`, `pa` and `stat` on a BLOW5 of the reads of _refcases.oracle_reads
  fuzz     the same for `event -c`, `event`, `stat` and `pa` on a BLOW5 of _refcases.fuzz_reads; the `stat` stdout
           also as text (ref_fuzz_<kind>_stat.txt)
  svbzd_grid, svbzd_reads
           sha256 of each svb-zd stream the reference's slow5lib stores for _refcases.svbzd_grid / svbzd_reads
           (read back from the BLOW5 blow5_write makes; blow5_dump must give the samples back)
Run from the repository root with oracle/_ref built; commit the outputs."""
import hashlib
import json
import os
import struct
import subprocess
import sys
import tempfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
import _refcases  # noqa: E402
from _blow5 import write_blow5  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
sha = lambda b: hashlib.sha256(b).hexdigest()


def ref_stdout(args, path):
    return subprocess.run([os.path.join(REF, "sigtk")] + args + [path], check=True, stdout=subprocess.PIPE,
                          stderr=subprocess.DEVNULL).stdout


def ref_streams(raws, tmp):
    """the svb-zd streams the reference's slow5lib writes for `raws`, checked against its own decode"""
    path = os.path.join(tmp, "svb.blow5")
    dump = b"".join(struct.pack("<I", 4) + b"r%03d" % i + struct.pack("<Qddd", len(r), 8192.0, 0.0, 1400.0) +
                    np.asarray(r, np.int16).tobytes() for i, r in enumerate(raws))
    subprocess.run([os.path.join(REF, "blow5_write"), path, "genomic_dna"], input=dump, check=True)
    d = open(path, "rb").read()
    assert d[:6] == b"BLOW5\x01" and d[9] == 1 and d[14] == 1, "expected zlib records and svb-zd signals"
    at = 68 + struct.unpack_from("<I", d, 64)[0]
    streams = []
    while d[at:at + 5] != b"5WOLB":
        n = struct.unpack_from("<Q", d, at)[0]
        rec = zlib.decompress(d[at + 8:at + 8 + n])
        at += 8 + n
        p = 2 + struct.unpack_from("<H", rec, 0)[0] + 4 + 32
        nb = struct.unpack_from("<Q", rec, p)[0]
        streams.append(rec[p + 8:p + 8 + nb])
    back = subprocess.run([os.path.join(REF, "blow5_dump"), path], check=True, stdout=subprocess.PIPE).stdout
    p = 0
    for r in raws:
        p += 4 + 4
        n = struct.unpack_from("<Q", back, p)[0]
        p += 32
        assert np.array_equal(np.frombuffer(back, np.int16, n, p), r)
        p += 2 * n
    assert len(streams) == len(raws)
    return streams


def main():
    out = {"oracle": {}, "fuzz": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for rna_flag, seed in _refcases.ORACLE_CASES:
            path = os.path.join(tmp, "oracle.blow5")
            write_blow5(path, "rna" if rna_flag else "genomic_dna", _refcases.oracle_reads(rna_flag, seed))
            out["oracle"][f"{rna_flag}-{seed}"] = {m: sha(ref_stdout([m], path)) for m in ("event", "pa", "stat")}
        for kind in _refcases.FUZZ_KINDS:
            path = os.path.join(tmp, "fuzz.blow5")
            write_blow5(path, kind, _refcases.fuzz_reads(kind))
            res = {}
            for args in (["event", "-c"], ["event"], ["stat"], ["pa"]):
                b = ref_stdout(args, path)
                res[" ".join(args)] = sha(b)
                if args == ["stat"]:
                    open(os.path.join(HERE, f"ref_fuzz_{kind}_stat.txt"), "wb").write(b)
            out["fuzz"][kind] = res
        out["svbzd_grid"] = [sha(s) for s in ref_streams(_refcases.svbzd_grid(), tmp)]
        out["svbzd_reads"] = [sha(s) for s in ref_streams(_refcases.svbzd_reads(), tmp)]
    json.dump(out, open(os.path.join(HERE, "ref_outputs.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()

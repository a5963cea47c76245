"""Writes SLOW5 / BLOW5 files for the command-line and reader tests; by default as slow5lib does (zlib records,
svb-zd signals)."""
from __future__ import annotations

import struct
import zlib

import numpy as np

from sigtk_b200.synth import svbzd_encode

TYPES = "#char*\tuint32_t\tdouble\tdouble\tdouble\tdouble\tuint64_t\tint16_t*"
NAMES = "#read_id\tread_group\tdigitisation\toffset\trange\tsampling_rate\tlen_raw_signal\traw_signal"


def _header(experiment_type: str, aux: bool) -> str:
    kit = "sqk-rna002" if experiment_type == "rna" else "sqk-lsk109"
    return (f"@experiment_type\t{experiment_type}\n@sequencing_kit\t{kit}\n" +
            TYPES + ("\tuint8_t" if aux else "") + "\n" + NAMES + ("\tstart_mux" if aux else "") + "\n")


def write_blow5(path: str, experiment_type: str, reads, zlib_records: bool = True, svbzd: bool = True,
                aux: bool = False) -> None:
    """reads: (read_id, int16 samples, digitisation, offset, range) per record. The header names the experiment type
    and the sequencing kit of an R9 pore, which decide the DNA / RNA parameters of the commands. aux adds a uint8
    auxiliary column (start_mux) after the primary ones."""
    text = _header(experiment_type, aux).encode()
    head = b"BLOW5\x01" + bytes([0, 2, 0, int(zlib_records)]) + struct.pack("<I", 1) + bytes([int(svbzd)])  # 0.2.0
    with open(path, "wb") as f:
        f.write(head.ljust(64, b"\0") + struct.pack("<I", len(text)) + text)
        for k, (rid, raw, dig, off, rng) in enumerate(reads):
            rid = rid.encode()
            raw = np.asarray(raw, dtype=np.int16)
            sig = svbzd_encode(raw).tobytes() if svbzd else raw.tobytes()
            n = len(sig) if svbzd else len(raw)
            rec = struct.pack("<H", len(rid)) + rid + struct.pack("<IddddQ", 0, dig, off, rng, 4000.0, n) + sig
            if aux:
                rec += bytes([k % 5])
            rec = zlib.compress(rec) if zlib_records else rec
            f.write(struct.pack("<Q", len(rec)) + rec)
        f.write(b"5WOLB")


def write_slow5(path: str, experiment_type: str, reads, aux: bool = False) -> None:
    """the same records as SLOW5 text, with a second read group that has no experiment type ('.')"""
    kit = "sqk-rna002" if experiment_type == "rna" else "sqk-lsk109"
    with open(path, "w") as f:
        f.write(f"#slow5_version\t0.2.0\n#num_read_groups\t2\n@experiment_type\t{experiment_type}\t.\n"
                f"@sequencing_kit\t{kit}\t{kit}\n" + TYPES + ("\tuint8_t" if aux else "") + "\n" + NAMES +
                ("\tstart_mux" if aux else "") + "\n")
        for k, (rid, raw, dig, off, rng) in enumerate(reads):
            f.write(f"{rid}\t{k % 2}\t{float(dig)!r}\t{float(off)!r}\t{float(rng)!r}\t4000\t{len(raw)}\t" +
                    ",".join(str(int(x)) for x in raw) + (f"\t{k % 5}" if aux else "") + "\n")


def npz_reads(d):
    """the records of a tests/golden/*.npz (read_ids, samples, read_off, digitisation, offset, range)"""
    return [(str(d["read_ids"][r]), d["samples"][int(d["read_off"][r]):int(d["read_off"][r + 1])],
             float(d["digitisation"][r]), float(d["offset"][r]), float(d["range"][r]))
            for r in range(len(d["read_ids"]))]

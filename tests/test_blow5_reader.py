"""The SLOW5 / BLOW5 reader of the command line (cli/blow5.c) through a small C driver (tests/tools/blow5_read.c):
every record layout it accepts gives back the stored reads, in file order and by read id, and malformed files are
errors. CPU only."""
import os
import struct
import subprocess

import numpy as np
import pytest

from _blow5 import npz_reads, write_blow5, write_slow5

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("blow5_read") / "blow5_read")
    subprocess.check_call(["gcc", "-O1", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "cli"),
                           os.path.join(ROOT, "tests", "tools", "blow5_read.c"), os.path.join(ROOT, "cli", "blow5.c"),
                           "-lz", "-o", exe])
    return exe


@pytest.fixture(scope="module")
def reads():
    return npz_reads(np.load(os.path.join(G, "synth_rna.npz")))


def read_all(driver, path, ids=()):
    p = subprocess.run([driver, path, *ids], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    out, b, at = [], p.stdout, 0
    while at < len(b):
        idl = struct.unpack_from("<I", b, at)[0]
        rid = b[at + 4:at + 4 + idl].decode()
        at += 4 + idl
        n, dig, off, rng = struct.unpack_from("<Qddd", b, at)
        at += 32
        out.append((rid, np.frombuffer(b, np.int16, n, at).copy(), dig, off, rng))
        at += 2 * n
    return p.returncode, out, p.stderr.decode()


def same(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g[0] == w[0] and g[2:] == tuple(w[2:]) and np.array_equal(g[1], w[1]), w[0]


@pytest.mark.parametrize("fmt", ["blow5-zlib-svbzd", "blow5-none-svbzd", "blow5-zlib-raw", "blow5-none-raw-aux",
                                 "slow5", "slow5-aux"])
def test_layouts_give_back_the_reads(driver, reads, tmp_path, fmt):
    path = str(tmp_path / ("reads.slow5" if fmt.startswith("slow5") else "reads.blow5"))
    if fmt.startswith("slow5"):
        write_slow5(path, "rna", reads, aux=fmt.endswith("aux"))
    else:
        write_blow5(path, "rna", reads, zlib_records="zlib" in fmt, svbzd="svbzd" in fmt, aux=fmt.endswith("aux"))
    rc, got, err = read_all(driver, path)
    assert rc == 0
    same(got, reads)
    assert "experiment_type[0]=rna" in err
    assert ("experiment_type[1]=(none)" in err) if fmt.startswith("slow5") else True
    pick = [reads[5][0], reads[0][0], reads[11][0]]
    rc, got, _ = read_all(driver, path, pick)
    assert rc == 0
    same(got, [reads[5], reads[0], reads[11]])
    assert read_all(driver, path, ["no-such-read"])[0] == 3


def test_the_stored_blow5_files(driver):
    for name in ("sp1_dna", "synth_rna"):
        rc, got, _ = read_all(driver, os.path.join(G, name + ".blow5"))
        assert rc == 0
        same(got, npz_reads(np.load(os.path.join(G, name + ".npz"))))


def test_malformed_files_are_errors(driver, reads, tmp_path):
    good = str(tmp_path / "good.blow5")
    write_blow5(good, "rna", reads[:3])
    data = open(good, "rb").read()
    for k, bad in enumerate([data[:-1], data[:-20], data[:100], b"BLOW4" + data[5:]]):
        path = str(tmp_path / f"bad{k}.blow5")
        open(path, "wb").write(bad)
        assert read_all(driver, path)[0] != 0, k
    flipped = bytearray(data)
    flipped[len(data) // 2] ^= 0xFF          # inside a zlib record: its checksum fails
    path = str(tmp_path / "flipped.blow5")
    open(path, "wb").write(bytes(flipped))
    assert read_all(driver, path)[0] == 4
    other = str(tmp_path / "reads.txt")      # neither .slow5 nor .blow5
    open(other, "wb").write(data)
    assert read_all(driver, other)[0] == 1
    for field in ("digitisation", "offset", "range", "samples"):
        path = str(tmp_path / f"bad_{field}.slow5")
        write_slow5(path, "rna", reads[:2])
        lines = open(path).read().split("\n")
        col = lines[6].split("\t")
        k = {"digitisation": 2, "offset": 3, "range": 4, "samples": 7}[field]
        col[k] += "x"
        lines[6] = "\t".join(col)
        open(path, "w").write("\n".join(lines))
        assert read_all(driver, path)[0] == 4, field

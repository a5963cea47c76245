"""The drop-in command line (cli/sigtk: C99 host + libsigtk_b200.so) against the stdout of the compiled,
unmodified reference (fixtures in tests/golden/, made by make_golden.py). Byte for byte."""
import gzip
import hashlib
import json
import os
import shutil
import subprocess

import pytest
import _refcases
from _blow5 import npz_reads, write_blow5

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "cli", "sigtk")
SHA = json.load(open(os.path.join(G, "sha256.json")))


def run(args, **kw):
    assert os.path.exists(CLI), "cli/sigtk is built by __graft_entry__.build()"
    return subprocess.run([CLI] + args, check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, **kw)


@pytest.fixture(scope="module")
def sp1(tmp_path_factory):
    d = tmp_path_factory.mktemp("blow5")
    shutil.copy(os.path.join(G, "sp1_dna.blow5"), d / "sp1_dna.blow5")  # the tests run on a copy, never on the tree
    return str(d / "sp1_dna.blow5")


RNA = os.path.join(G, "synth_rna.blow5")


def test_event_compact_dna(sp1):
    p = run(["event", "-c", sp1])
    assert p.stdout == open(os.path.join(G, "ref_sp1_event_c.txt"), "rb").read()
    assert b"DNA data detected." in p.stderr and b"Real time:" in p.stderr


def test_event_long_pa_stat_dna_full_output_hashes(sp1):
    assert hashlib.sha256(run(["event", sp1]).stdout).hexdigest() == SHA["sp1_event"]
    assert hashlib.sha256(run(["pa", sp1]).stdout).hexdigest() == SHA["sp1_pa"]
    out = run(["stat", sp1]).stdout
    assert out == open(os.path.join(G, "ref_sp1_stat.txt"), "rb").read()
    assert hashlib.sha256(out).hexdigest() == SHA["sp1_stat"]


def test_event_by_read_id_equals_the_reference_golden_file(sp1):
    """scripts/test.sh:70-72 of the reference: one read by id, long form, vs test/event_dna.exp (stale header line)"""
    p = run(["event", sp1, "05d90f17-f4a6-4349-924c-3ffd3457a99d"])
    exp = open(os.path.join(G, "event_dna.exp"), "rb").read().split(b"\n", 1)[1]
    assert p.stdout.split(b"\n", 1)[1] == exp
    assert b"Read ID 05d90f17-f4a6-4349-924c-3ffd3457a99d" in p.stderr


def test_read_ids_in_argv_order_and_options_after_positionals(sp1):
    ids = [l.split(b"\t")[0].decode() for l in open(os.path.join(G, "ref_sp1_event_c.txt"), "rb").read().splitlines()[1:]]
    pick = [ids[7], ids[2], ids[40]]
    p = run(["event", sp1] + pick + ["-n", "-c"])
    got = [l.split(b"\t")[0].decode() for l in p.stdout.splitlines()]
    assert got == pick


def test_rna_long_compact_stat_pa():
    assert run(["event", RNA]).stdout == gzip.open(os.path.join(G, "ref_rna_event.txt.gz"), "rb").read()
    p = run(["event", "-c", RNA])
    assert p.stdout == open(os.path.join(G, "ref_rna_event_c.txt"), "rb").read()
    assert b"RNA data detected." in p.stderr
    assert run(["stat", RNA]).stdout == open(os.path.join(G, "ref_rna_stat.txt"), "rb").read()
    assert hashlib.sha256(run(["pa", RNA]).stdout).hexdigest() == SHA["rna_pa"]


def test_small_batches_give_the_same_bytes(sp1):
    """many batches in flight (slots of 1M samples... forced down to a few reads per batch)"""
    p = run(["event", "-c", "--batch-samples", "20000", sp1])
    assert p.stdout == open(os.path.join(G, "ref_sp1_event_c.txt"), "rb").read()


def test_no_header_version_help_and_errors(sp1):
    p = run(["stat", "-n", sp1])
    assert p.stdout == open(os.path.join(G, "ref_sp1_stat.txt"), "rb").read().split(b"\n", 1)[1]
    assert run(["--version"]).stdout == b"sigtk 0.2.0\n"
    assert run(["event", "-h"]).stdout.startswith(b"Usage: sigtk event reads.blow5")
    r = subprocess.run([CLI, "event"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and r.stderr.startswith(b"Usage: sigtk event")
    r = subprocess.run([CLI, "event", "/nonexistent.blow5"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"cannot open /nonexistent.blow5" in r.stderr
    r = subprocess.run([CLI, "sref", sp1], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"outside the B200 raw-signal hot path" in r.stderr


def test_ent_equals_the_reference_stdout(sp1, tmp_path):
    """`sigtk ent` (src/ent.c): stdout of the compiled reference on the DNA file, the synthetic RNA file and a BLOW5 of
    reads with wide / wrapped / single-bin histograms (tests/golden/ent_adversarial.npz); its own option set"""
    import numpy as np
    exp = open(os.path.join(G, "ref_sp1_ent.txt"), "rb").read()
    p = run(["ent", sp1])
    assert p.stdout == exp
    assert b"data detected" not in p.stderr and b"Real time:" in p.stderr  # entmain does not inspect the header
    assert run(["ent", "--cpu-decode", "--batch-samples", "30000", sp1]).stdout == exp
    assert run(["ent", "--no-header", sp1]).stdout == exp.split(b"\n", 1)[1]
    assert run(["ent", RNA]).stdout == open(os.path.join(G, "ref_rna_ent.txt"), "rb").read()
    assert run(["ent", "-h"]).stdout.startswith(b"Usage: sigtk ent a.blow5\n")
    r = subprocess.run([CLI, "ent", sp1, "some-read-id"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and r.stderr.startswith(b"Usage: sigtk ent a.blow5\n")
    r = subprocess.run([CLI, "ent", "/nonexistent.blow5"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"Error in opening file" in r.stderr
    path = str(tmp_path / "ent_adv.blow5")
    write_blow5(path, "genomic_dna", npz_reads(np.load(os.path.join(G, "ent_adversarial.npz"))))
    assert run(["ent", path]).stdout == open(os.path.join(G, "ref_ent_adversarial.txt"), "rb").read()


@pytest.mark.parametrize("kind", ["dna", "rna"])
def test_jnn_equals_the_reference_stdout(sp1, tmp_path, kind):
    """`sigtk jnn` and `jnn -c` (src/jnn.c): stdout of the compiled reference on the DNA file / the synthetic RNA file
    and on a BLOW5 of reads with stalls (tests/golden/jnn_stalls_*.npz)"""
    import numpy as np
    path, tag = (sp1, "sp1") if kind == "dna" else (RNA, "rna")
    p = run(["jnn", path])
    assert p.stdout == open(os.path.join(G, f"ref_{tag}_jnn.txt"), "rb").read()
    assert (b"RNA data detected." if kind == "rna" else b"DNA data detected.") in p.stderr
    assert run(["jnn", "-c", "--batch-samples", "30000", path]).stdout == open(os.path.join(G, f"ref_{tag}_jnn_c.txt"), "rb").read()
    assert run(["jnn", "--cpu-decode", "-n", path]).stdout == open(os.path.join(G, f"ref_{tag}_jnn.txt"), "rb").read().split(b"\n", 1)[1]
    path = str(tmp_path / "stalls.blow5")
    write_blow5(path, "rna" if kind == "rna" else "genomic_dna", npz_reads(np.load(os.path.join(G, f"jnn_stalls_{kind}.npz"))))
    assert run(["jnn", path]).stdout == open(os.path.join(G, f"ref_jnn_stalls_{kind}.txt"), "rb").read()
    assert run(["jnn", "-c", path]).stdout == open(os.path.join(G, f"ref_jnn_stalls_{kind}_c.txt"), "rb").read()


@pytest.mark.parametrize("kind", ["dna", "rna"])
def test_prefix_equals_the_reference_stdout(sp1, tmp_path, kind):
    """`sigtk prefix` and `prefix --print-stat` (src/cfunc.c:169-234): the reference's own golden test/prefix_dna.exp,
    the stdout of the compiled reference on the DNA file / the synthetic RNA file and on a BLOW5 of reads with adaptor
    and poly-A like stretches (tests/golden/prefix_adaptor_*.npz)"""
    import numpy as np
    path, tag = (sp1, "sp1") if kind == "dna" else (RNA, "rna")
    exp_stat = open(os.path.join(G, f"ref_{tag}_prefix_stat.txt"), "rb").read()
    p = run(["prefix", "--print-stat", path])
    assert p.stdout == exp_stat
    assert (b"RNA data detected." if kind == "rna" else b"DNA data detected.") in p.stderr
    if kind == "dna":
        assert run(["prefix", path]).stdout == open(os.path.join(G, "prefix_dna.exp"), "rb").read()
    assert run(["prefix", "--print-stat", "--cpu-decode", "--batch-samples", "60000", "-n", path]).stdout == exp_stat.split(b"\n", 1)[1]
    path = str(tmp_path / "adaptor.blow5")
    write_blow5(path, "rna" if kind == "rna" else "genomic_dna", npz_reads(np.load(os.path.join(G, f"prefix_adaptor_{kind}.npz"))))
    assert run(["prefix", path]).stdout == open(os.path.join(G, f"ref_prefix_adaptor_{kind}.txt"), "rb").read()
    assert run(["prefix", "--print-stat", path]).stdout == open(os.path.join(G, f"ref_prefix_adaptor_{kind}_stat.txt"), "rb").read()


def test_two_gpus_same_bytes(sp1):
    import ctypes as C
    from sigtk_b200 import _lib
    if _lib.load().sgpu_device_count() < 2:
        pytest.skip("needs two GPUs")
    p = run(["event", "-c", "--gpus", "2", "--batch-samples", "50000", sp1])
    assert p.stdout == open(os.path.join(G, "ref_sp1_event_c.txt"), "rb").read()


def test_cpu_decode_flag_gives_the_same_bytes(sp1):
    """sp1_dna.blow5 is zlib + svb-zd: by default the svb-zd streams are decoded on the GPU (svbzd.cu); --cpu-decode
    decodes them on the host threads (cli/blow5.c). Both equal the reference."""
    exp = open(os.path.join(G, "ref_sp1_event_c.txt"), "rb").read()
    assert run(["event", "-c", "--cpu-decode", sp1]).stdout == exp
    p = run(["event", "-c", sp1], env=dict(os.environ, SIGTK_PROFILE="1"))
    assert p.stdout == exp and b"signal decode: GPU (svb-zd)" in p.stderr
    assert hashlib.sha256(run(["pa", "--cpu-decode", sp1]).stdout).hexdigest() == SHA["sp1_pa"]
    assert run(["stat", "--cpu-decode", "--batch-samples", "30000", sp1]).stdout == open(
        os.path.join(G, "ref_sp1_stat.txt"), "rb").read()
    assert run(["stat", "--batch-samples", "30000", sp1]).stdout == open(os.path.join(G, "ref_sp1_stat.txt"), "rb").read()


REF_OUT = json.load(open(os.path.join(G, "ref_outputs.json")))


@pytest.mark.parametrize("kind", _refcases.FUZZ_KINDS)
def test_adversarial_blow5_against_the_reference_binary(tmp_path, kind):
    """a BLOW5 (zlib + svb-zd) of reads with glitches (pA <= 0), flat stretches, ramps, steps and saturation
    (_refcases.fuzz_reads); stdout of `event`, `event -c`, `stat` and `pa` must equal the stdout of the compiled
    unmodified reference on the same file, byte for byte (sha256 in tests/golden/ref_outputs.json, the `stat`
    stdout in ref_fuzz_<kind>_stat.txt; made by make_ref_outputs.py)"""
    path = str(tmp_path / "fuzz.blow5")
    write_blow5(path, kind, _refcases.fuzz_reads(kind))
    assert run(["stat", path]).stdout == open(os.path.join(G, f"ref_fuzz_{kind}_stat.txt"), "rb").read()
    for args in (["event", "-c"], ["event"], ["stat"], ["pa"]):
        ours = run(args + [path])
        assert hashlib.sha256(ours.stdout).hexdigest() == REF_OUT["fuzz"][kind][" ".join(args)], args

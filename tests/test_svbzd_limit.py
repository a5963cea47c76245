"""The bound that decides which reads the svb-zd encoder takes (SGPU_SVBZD_MAX_BYTES in include/sigtk_b200.h, used by
sgpu_submit and sgpu_encode_svbzd_device): the longest stream of n int16 samples is 4 + ceil(n/4) + 3n bytes, and
comp_len's uint32_t holds it exactly up to n = 1,321,528,397. Compiled with the host C compiler; no GPU."""
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIMIT = 1_321_528_397
NS = [0, 1, 2, 3, 4, 5, 1023, 1024, 1025, 2_000_000, LIMIT - 1, LIMIT, LIMIT + 1, LIMIT + 2, (1 << 31) - 1, 1 << 31,
      (1 << 32) - 1]


def test_stream_bound_and_limit(tmp_path):
    src = tmp_path / "bound.c"
    src.write_text('#include <inttypes.h>\n#include <stdio.h>\n#include "sigtk_b200.h"\n'
                   'int main(void) {\n  static const uint64_t ns[] = {' + ", ".join(f"{n}ull" for n in NS) + '};\n'
                   '  for (unsigned k = 0; k < sizeof ns / sizeof ns[0]; k++)\n'
                   '    printf("%" PRIu64 " %d\\n", (uint64_t)SGPU_SVBZD_MAX_BYTES(ns[k]),\n'
                   '           SGPU_SVBZD_MAX_BYTES(ns[k]) <= 0xffffffffull);\n  return 0;\n}\n')
    exe = tmp_path / "bound"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src), "-o",
                           str(exe)])
    rows = [ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines()]
    assert len(rows) == len(NS)
    for n, (bound, fits) in zip(NS, rows):
        assert int(bound) == 4 + (n + 3) // 4 + 3 * n, n
        assert int(fits) == (n <= LIMIT), n
    assert 4 + (LIMIT + 3) // 4 + 3 * LIMIT == 2**32 - 1


def test_bound_holds_for_every_stream(tmp_path):
    """no int16 signal takes more: every value is at most 3 bytes (z = zigzag(d) <= 131070 < 2^24)"""
    from sigtk_b200 import synth
    rng = np.random.default_rng(3)
    for n in (0, 1, 5, 1000):
        worst = np.tile(np.array([-32768, 32767], np.int16), n // 2 + 1)[:n]
        for raw in (worst, rng.integers(-32768, 32768, n).astype(np.int16)):
            assert len(synth.svbzd_encode(raw)) <= 4 + (n + 3) // 4 + 3 * n
    # the first value, -32768 - 0, takes 2 bytes; each of the other 999 takes 3
    assert len(synth.svbzd_encode(np.tile(np.array([-32768, 32767], np.int16), 500))) == 4 + 250 + 2 + 3 * 999

"""Device time of `sigtk prefix` (SGPU_WANT_PREFIX: prefix_walk + prefix_median) with the caller's own sets
(sgpu_set_prefix).

Batches, device resident (sgpu_run_device, SGPU_WANT_PREFIX only, rna = 1 so that the poly-A walk runs):
  bench    bench.py's synthetic batch (the first 16,384 reads of the named set, generated on the GPU)
  adaptor  2,048 direct-RNA-like reads of 20,000 to 150,000 samples (seeded on the host, tests/_prefix_ref.set_read
           with the R9 sets): a low adaptor stretch, a poly-A plateau about 30 pA above it, then the transcript
Configurations, alternated run by run so that all see the same card state:
  default      no set (JNNV2_RNA_R9_ADAPTOR and JNNV1_R9_POLYA, SGPU_PARAM_PORE = 0)
  r9_set       those sets given explicitly: the same kernel with the same arguments
  rna004_set   JNNV2_RNA_RNA004_ADAPTOR and JNNV1_R9_POLYA given explicitly: the same kernel
  window_2667  the adaptor window scaled to 4 kHz (2667, not a multiple of 8): prefix_set_walk_kernel
  automaton    a poly-A set on the automaton route (250, 1.0, 32, 200, 40)
  exact        a poly-A set on the exact route, error = corrector (250, 1.0, 30, 200, 30)
Each run is timed with the context's stage timers (CUDA events around each kernel group, SGPU_F_STAGE_TIMERS) after
--warmup runs of every configuration; the lines give the median, min and max over --iters runs of the `prefix` stage,
the reads with an adaptor and with a poly-A and, for the explicit reference sets, whether all outputs equal the
default's (r9_set) or PORE = 1's (rna004_set).

--root DIR times the package and library of another tree (e.g. the parent commit's, built in DIR) with the same
batches; such a tree without sgpu_set_prefix runs the default configuration only (--configs default). Prints one JSON
line per (batch, configuration), and the card's name, power limit and max SM clock.

    python tools/prefix_set_time.py [--iters 20] [--warmup 3] [--root DIR] [--configs default,r9_set] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_ROOT = os.path.abspath(sys.argv[sys.argv.index("--root") + 1]) if "--root" in sys.argv else ROOT
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, PKG_ROOT)  # the package (and library) timed

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import live_time  # noqa: E402
import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import _lib as _sl  # noqa: E402
from sigtk_b200 import synth  # noqa: E402

R9 = ((2000, 0.5, 1500, 2000, 200000), (250, 1.0, 30, 200, 50))
CONFIGS = {
    "default": None,
    "r9_set": R9,
    "rna004_set": ((2000, 0.7, 1500, 500, 200000), R9[1]),
    "window_2667": ((2667, 0.6, 2000, 667, 266667), R9[1]),
    "automaton": (R9[0], (250, 1.0, 32, 200, 40)),
    "exact": (R9[0], (250, 1.0, 30, 200, 30)),
}


def adaptor_batch(dev, n_reads=2048, seed=23):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _prefix_ref import set_read
    rng = np.random.default_rng(seed)
    reads = [set_read(k, seed, R9, n=int(rng.integers(20000, 150000))) for k in range(n_reads)]
    lens = np.array([len(r[0]) for r in reads], np.int64)
    off = np.zeros(n_reads + 1, np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    raw = np.zeros(int(off[-1]), np.int16)
    for r, rd in enumerate(reads):
        raw[off[r]:off[r] + lens[r]] = rd[0]
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)  # noqa: E731
    return {"samples": t(raw), "read_off": t(off), "read_len": t(lens.astype(np.int32)),
            "offset": t(np.array([np.float32(rd[2]) for rd in reads], np.float32)),
            "unit": t(np.array([np.float32(rd[3]) / np.float32(rd[1]) for rd in reads], np.float32)),
            "span": int(off[-1]), "n_reads": n_reads}


def time_batch(name, b, configs, a):
    span, n = b["span"], b["n_reads"]
    lines = []
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS) as c:
        st = torch.cuda.current_stream().cuda_stream

        def run(p, pore=0):
            if p is not None or hasattr(c, "set_prefix"):
                c.set_prefix(None if p is None else sg.Prefix(sg.Adaptor(*p[0]), sg.Polya(*p[1])))
            c.set_param(_sl.PARAM_PORE, pore)
            d = c.run_device(b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(),
                             b["offset"].data_ptr(), b["unit"].data_ptr(), n, span, 1, sg.WANT_PREFIX, st)
            stages = {s: ms for s, ms, _ in c.stage_times()}
            return d, stages

        def outputs(p, pore=0):
            d, _ = run(p, pore)
            torch.cuda.synchronize()
            assert c.counters()["status"] == 0
            return c.d2h(d.prefix_pos, np.int32, 4 * n).copy(), c.d2h(d.prefix_stat, np.float32, 6 * n).view(np.uint32).copy()

        outs = {cfg: outputs(CONFIGS[cfg]) for cfg in configs}
        pore1 = outputs(None, 1) if "rna004_set" in configs else None
        for _ in range(a.warmup):
            for cfg in configs:
                run(CONFIGS[cfg])
        t = {cfg: [] for cfg in configs}
        for _ in range(a.iters):
            for cfg in configs:
                t[cfg].append(run(CONFIGS[cfg])[1]["prefix"])
        for cfg in configs:
            ms = np.array(t[cfg])
            pos, _ = outs[cfg]
            line = {"batch": name, "config": cfg, "set": CONFIGS[cfg], "tree": a.root or "this", "reads": n,
                    "samples": span, "runs_timed": a.iters,
                    "prefix_ms": {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())},
                    "gsamples_per_s": span / float(np.median(ms)) / 1e6,
                    "adaptors": int((pos.reshape(n, 4)[:, 1] > 0).sum()),
                    "polyas": int((pos.reshape(n, 4)[:, 3] > 0).sum())}
            same_as = outs.get("default") if cfg == "r9_set" else pore1 if cfg == "rna004_set" else None
            if same_as is not None:
                line["outputs_equal_default"] = bool(all(np.array_equal(x, y) for x, y in zip(outs[cfg], same_as)))
            lines.append(line)
            print(json.dumps(line), flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--root", default="", help="a tree whose sigtk_b200 package and library to time instead")
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--batches", default="bench,adaptor")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    configs = a.configs.split(",")
    dev = torch.device("cuda:0")
    lines = [{"card": live_time.card()}]
    print(json.dumps(lines[0]), flush=True)
    for name in a.batches.split(","):
        if name == "bench":
            b = bench.device_batch(torch, dev, synth.read_lengths(bench.N_SET)[:a.reads], 0, synth.SEED, 0.1)
        else:
            b = adaptor_batch(dev)
        torch.cuda.synchronize()
        lines += time_batch(name, b, configs, a)
        del b
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "a") as f:
            for ln_ in lines:
                f.write(json.dumps(ln_) + "\n")


if __name__ == "__main__":
    main()

"""Device time of `sigtk jnn` (SGPU_WANT_JNN: jnn_moments + jnn_walk) with the caller's own parameters (sgpu_set_jnn).

Batches, device resident (sgpu_run_device, SGPU_WANT_JNN only):
  bench   bench.py's synthetic DNA batch (the first 16,384 reads of the named set, generated on the GPU)
  stalls  4,096 reads of about 40,000 samples (seeded on the host): noise around a level with flat stalls of 20 to
          3,000 samples, outliers inside half of them
Configurations, alternated run by run so that all see the same card state:
  default     no set (jnn_print's DNA set, chosen by rna = 0)
  dna_set     that set given explicitly (150, 0.25, 5, 50, 50, 0.75): the same route and kernel
  automaton   a custom set on the automaton route (188, 0.25, 4, 60, 50, 0.7)
  exact_corr  a set whose corrector acts (error >= corrector) (150, 0.25, 50, 50, 50, 0.75): jnn_exact_kernel
  exact_e40   error 40 (188, 0.25, 40, 60, 10, 0.7): jnn_exact_kernel
Each run is timed with the context's stage timers (CUDA events around each kernel group, SGPU_F_STAGE_TIMERS) after
--warmup runs of every configuration; the lines give the median, min and max over --iters runs of jnn_moments, of
jnn_walk and of their sum, the segments found and, for dna_set, whether they equal the default's.

--root DIR times the package and library of another tree (e.g. the parent commit's, built in DIR) with the same
batches; such a tree without sgpu_set_jnn runs the default configuration only (--configs default). Prints one JSON line per (batch, configuration), and the card's name, power limit and max SM clock.

    python tools/jnn_set_time.py [--iters 30] [--warmup 3] [--root DIR] [--configs default,dna_set] [--out FILE]
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
from sigtk_b200 import synth  # noqa: E402

CONFIGS = {
    "default": None,
    "dna_set": (150, 0.25, 5, 50, 50, 0.75),
    "automaton": (188, 0.25, 4, 60, 50, 0.7),
    "exact_corr": (150, 0.25, 50, 50, 50, 0.75),
    "exact_e40": (188, 0.25, 40, 60, 10, 0.7),
}


def stall_batch(dev, n_reads=4096, mean_len=40000, seed=17):
    rng = np.random.default_rng(seed)
    lens = rng.integers(mean_len // 2, 3 * mean_len // 2, n_reads).astype(np.int64)
    al = (lens + 7) // 8 * 8
    off = np.zeros(n_reads + 1, np.int64)
    off[1:] = np.cumsum(al)
    span = int(off[-1])
    raw = (rng.integers(300, 700, n_reads).repeat(al) + 60 * rng.standard_normal(span)).astype(np.int64)
    pos = 0
    while pos < span:  # stalls across the whole span (a stall may cross into the next read: still a stall there)
        stop = min(span, pos + int(rng.integers(20, 3000)))
        raw[pos:stop] = raw[pos] + rng.integers(-6, 7, stop - pos)
        if rng.integers(0, 2):
            raw[rng.integers(pos, stop, int(rng.integers(1, 40)))] += 400
        pos = stop + int(rng.integers(3, 2000))
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)  # noqa: E731
    return {"samples": t(np.clip(raw, -32768, 32767).astype(np.int16)), "read_off": t(off),
            "read_len": t(lens.astype(np.int32)), "offset": t(np.zeros(n_reads, np.float32)),
            "unit": t(np.full(n_reads, np.float32(1400.0) / np.float32(8192.0), np.float32)), "span": span,
            "n_reads": n_reads}


def time_batch(name, b, configs, a):
    span, n = b["span"], b["n_reads"]
    lines = []
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS) as c:
        st = torch.cuda.current_stream().cuda_stream

        def run(p):
            if p is not None or hasattr(c, "set_jnn"):
                c.set_jnn(None if p is None else sg.Jnn(*p))
            d = c.run_device(b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(),
                             b["offset"].data_ptr(), b["unit"].data_ptr(), n, span, 0, sg.WANT_JNN, st)
            stages = {s: ms for s, ms, _ in c.stage_times()}
            return d, stages

        segs = {}
        for cfg in configs:  # outputs of one run of each
            d, _ = run(CONFIGS[cfg])
            torch.cuda.synchronize()
            assert c.counters()["status"] == 0, cfg
            cnt = c.d2h(d.jnn_cnt, np.uint32, n)
            seg = c.d2h(d.jnn_seg, np.int32, 2 * ((span >> 5) + n + 1))
            segs[cfg] = (cnt, seg)
        for _ in range(a.warmup):
            for cfg in configs:
                run(CONFIGS[cfg])
        t = {cfg: [] for cfg in configs}
        for _ in range(a.iters):
            for cfg in configs:
                t[cfg].append(run(CONFIGS[cfg])[1])
        off = b["read_off"].cpu().numpy()
        for cfg in configs:
            mom = np.array([s["jnn_moments"] for s in t[cfg]])
            walk = np.array([s["jnn_walk"] for s in t[cfg]])
            tot = mom + walk
            cnt, seg = segs[cfg]
            line = {"batch": name, "config": cfg, "set": CONFIGS[cfg], "tree": a.root or "this", "reads": n,
                    "samples": span, "runs_timed": a.iters,
                    "jnn_moments_ms": {"median": float(np.median(mom)), "min": float(mom.min()), "max": float(mom.max())},
                    "jnn_walk_ms": {"median": float(np.median(walk)), "min": float(walk.min()), "max": float(walk.max())},
                    "total_ms_median": float(np.median(tot)),
                    "gsamples_per_s": span / float(np.median(tot)) / 1e6, "segments": int(cnt.sum())}
            if cfg == "dna_set" and "default" in segs:
                c0, s0 = segs["default"]
                line["segments_equal_default"] = bool(np.array_equal(cnt, c0) and all(
                    np.array_equal(seg[2 * ((int(off[r]) >> 5) + r):][:2 * int(cnt[r])],
                                   s0[2 * ((int(off[r]) >> 5) + r):][:2 * int(cnt[r])]) for r in range(n)))
            lines.append(line)
            print(json.dumps(line), flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--root", default="", help="a tree whose sigtk_b200 package and library to time instead")
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--batches", default="bench,stalls")
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
            b = stall_batch(dev)
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

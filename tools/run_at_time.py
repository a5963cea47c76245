"""Device time of runs on reads at any sample offset (sgpu_run_device_at, stage.cu) against sgpu_run_device on the
aligned layout, and of the gather itself (its stage "stage_reads").

Batches, device resident (int16 samples generated on the GPU by bench.device_batch):
  bench  bench.py's synthetic DNA batch: the first 16,384 reads of its set
  long   320 reads of 2,000,000 samples of the same generator
Each batch is also copied, on the device, into a packed tensor: the reads back to back without padding, the first at
element 1 of its allocation (so the base and most reads are misaligned). After --warmup runs of each, --iters rounds
alternate sgpu_run_device on the aligned batch and sgpu_run_device_at on the packed one (span = the aligned batch's, so
both runs pick the same chunk length), for events only and for all six products, each timed with CUDA events on the
stream it runs on. The outputs of the two runs are compared bit for bit before timing (the event table; with all
products also stat, ent, jnn counts, prefix positions and the pa of every 256th read). Both working sets exceed the 126 MB L2.

  rna_trimmed  the bench lengths generated as RNA-like reads (p_change 0.025) and run with the RNA parameters: a
               device-resident SGPU_WANT_PREFIX run, then the events of every read from its adaptor's (and poly-A's)
               end, read_off + start and read_len - start formed on the device, through sgpu_run_device_at.

"stage_reads" is the gather's stage from sgpu_stage_times (4 launches: count, scan, offsets, gather) in the timed
runs; its GB/s counts the bytes the gather must move, 2 B per sample read plus 2 B per staged sample written, over its
time, against the 7.7 TB/s of the B200's data sheet. Each line gives the card's name, power limit and max SM clock read
in the same call.

    python tools/run_at_time.py [--iters 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import live_time  # noqa: E402
import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import synth  # noqa: E402

ALL = sg.WANT_EVENTS | sg.WANT_PA | sg.WANT_STAT | sg.WANT_ENT | sg.WANT_JNN | sg.WANT_PREFIX
PEAK_GBS = 7700.0


def timed(fn, st):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b)


def packed_copy(b, dev):
    """the batch's reads back to back without padding, from element 1 of a new tensor; -> (slice, read_off i64)"""
    lens = torch.from_numpy(b["host_len"].astype(np.int64)).to(dev)
    n, total = b["n_reads"], b["n_samples"]
    poff = torch.zeros(n, dtype=torch.int64, device=dev)
    poff[1:] = torch.cumsum(lens, 0)[:-1]
    rid = torch.repeat_interleave(torch.arange(n, device=dev), lens, output_size=total)
    src = b["read_off"][:-1][rid] + (torch.arange(total, device=dev) - poff[rid])
    del rid
    big = torch.zeros(total + 2, dtype=torch.int16, device=dev)
    big[1:1 + total] = b["samples"][src]
    del src
    return big[1:1 + total], poff


def outputs(c, d, n, off, lens, span, want):
    """host copies of the outputs that are compared (pa through the layout)"""
    o = {"ev_off": c.d2h(d.ev_off, np.uint64, n + 1)}
    ne = int(o["ev_off"][-1])
    o["ev_start"] = c.d2h(d.ev_start, np.uint32, ne)
    o["ev_mean"] = c.d2h(d.ev_mean, np.uint32, ne)
    o["ev_stdv"] = c.d2h(d.ev_stdv, np.uint32, ne)
    if want & sg.WANT_STAT:
        o["stat"] = c.d2h(d.stat, np.uint32, 6 * n)
    if want & sg.WANT_JNN:
        o["jnn_cnt"] = c.d2h(d.jnn_cnt, np.uint32, n)
    if want & sg.WANT_PREFIX:
        o["prefix_pos"] = c.d2h(d.prefix_pos, np.int32, 4 * n)
    if want & sg.WANT_ENT:
        o["ent"] = c.d2h(d.ent, np.uint64, 3 * n)
    if want & sg.WANT_PA:  # (every 256th read)
        flat = c.d2h(d.pa, np.uint32, span)
        o["pa"] = np.concatenate([flat[int(off[r]): int(off[r]) + int(lens[r])] for r in range(0, n, 256)])
    return o


def stage_reads(c):
    st = [s for s in c.stage_times() if s[0] == "stage_reads"]
    assert st, "no stage_reads stage"
    return st[0][1]


def ms_stats(ms):
    ms = np.array(ms)
    return {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())}


def time_batch(name, b, a, card, dev):
    n, span, n_samp = b["n_reads"], b["span"], b["n_samples"]
    st = torch.cuda.current_stream()
    t, poff = packed_copy(b, dev)
    torch.cuda.synchronize()
    lines = []
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS) as c:
        al = (b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(), b["offset"].data_ptr(),
              b["unit"].data_ptr())
        for want, wname in ((sg.WANT_EVENTS, "events"), (ALL, "all")):
            def aligned():
                return c.run_device(*al, n, span, 0, want, st.cuda_stream)

            def at():
                return c.run_device_at(t.data_ptr(), t.numel(), poff.data_ptr(), al[2], al[3], al[4], n, span, 0, want,
                                       st.cuda_stream)

            ref = outputs(c, aligned(), n, b["host_off"], b["host_len"], span, want)
            d, soff = at()
            got = outputs(c, d, n, c.d2h(soff, np.uint64, n + 1), b["host_len"], span, want)
            assert c.counters()["status"] == 0
            for k in ref:
                assert np.array_equal(ref[k], got[k]), f"{name} {wname}: {k} differs"
            del ref, got
            for _ in range(a.warmup):
                aligned()
                at()
            ta, tb, ts = [], [], []
            for _ in range(a.iters):
                ta.append(timed(aligned, st))
                tb.append(timed(at, st))
                ts.append(stage_reads(c))
            med_a, med_b, med_s = float(np.median(ta)), float(np.median(tb)), float(np.median(ts))
            moved = 2 * n_samp + 2 * span
            lines.append({"batch": name, "want": wname, "reads": n, "samples": n_samp, "runs_timed": a.iters,
                          "layout_at": "packed, no padding, base at element 1",
                          "run_device_aligned_ms": ms_stats(ta), "run_device_at_ms": ms_stats(tb),
                          "stage_reads_ms": ms_stats(ts), "at_over_aligned": med_b / med_a,
                          "stage_reads_share_of_at": med_s / med_b,
                          "stage_reads_gb_per_s": moved / med_s / 1e6,
                          "stage_reads_share_of_7700_gb_per_s": moved / med_s / 1e6 / PEAK_GBS,
                          "checked": "outputs of both runs bit-identical", "card": card})
    del t, poff
    return lines


def time_trimmed(b, a, card, dev):
    n, span, n_samp = b["n_reads"], b["span"], b["n_samples"]
    st = torch.cuda.current_stream()
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS) as c:
        al = (b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(), b["offset"].data_ptr(),
              b["unit"].data_ptr())
        d = c.run_device(*al, n, span, 1, sg.WANT_PREFIX, st.cuda_stream)
        pos = torch.from_numpy(c.d2h(d.prefix_pos, np.int32, 4 * n).reshape(n, 4).astype(np.int64)).to(dev)
        start = torch.where(pos[:, 1] > 0, pos[:, 1] + torch.where(pos[:, 3] > 0, pos[:, 3], 0), 0)
        start = torch.minimum(start, b["read_len"].to(torch.int64))
        off2 = b["read_off"][:-1] + start
        len2 = (b["read_len"].to(torch.int64) - start).to(torch.int32)
        trimmed = int((start > 0).sum())
        kept = int(len2.to(torch.int64).sum())

        def at():
            return c.run_device_at(b["samples"].data_ptr(), b["samples"].numel(), off2.data_ptr(), len2.data_ptr(),
                                   al[3], al[4], n, span, 1, sg.WANT_EVENTS, st.cuda_stream)

        def aligned():
            return c.run_device(*al, n, span, 1, sg.WANT_EVENTS, st.cuda_stream)

        at()
        torch.cuda.synchronize()
        assert c.counters()["status"] == 0
        for _ in range(a.warmup):
            aligned()
            at()
        ta, tb, ts = [], [], []
        for _ in range(a.iters):
            ta.append(timed(aligned, st))
            tb.append(timed(at, st))
            ts.append(stage_reads(c))
    med_s = float(np.median(ts))
    moved = 2 * kept + 2 * span
    return [{"batch": "rna_trimmed", "want": "events", "reads": n, "samples": n_samp, "reads_trimmed": trimmed,
             "samples_after_trimming": kept, "runs_timed": a.iters,
             "run_device_untrimmed_ms": ms_stats(ta), "run_device_at_trimmed_ms": ms_stats(tb),
             "stage_reads_ms": ms_stats(ts), "stage_reads_gb_per_s": moved / med_s / 1e6,
             "stage_reads_share_of_7700_gb_per_s": moved / med_s / 1e6 / PEAK_GBS, "card": card}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    card = live_time.card()
    lines = []
    for name in ("bench", "long", "rna_trimmed"):
        lens = np.full(320, 2_000_000, np.int64) if name == "long" else synth.read_lengths(bench.N_SET)[:16384]
        b = bench.device_batch(torch, dev, lens, 0, synth.SEED, 0.025 if name == "rna_trimmed" else 0.1)
        torch.cuda.synchronize()
        new = time_trimmed(b, a, card, dev) if name == "rna_trimmed" else time_batch(name, b, a, card, dev)
        for ln_ in new:
            print(json.dumps(ln_), flush=True)
        lines += new
        del b
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "a") as f:
            for ln_ in lines:
                f.write(json.dumps(ln_) + "\n")


if __name__ == "__main__":
    main()

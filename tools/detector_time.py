"""Device time of event detection with the caller's own detector parameters (sgpu_set_detector).

Batches: bench.py's synthetic DNA batch (the first 16,384 reads of the named set, generated on the GPU), run from
device memory (sgpu_run_device, SGPU_WANT_EVENTS) in three configurations, alternated run by run so that all three see
the same card state:
  default   no set: the chunk walker and the fast emitter
  dna_set   the reference's DNA set given explicitly: the general route (witness-checked scan of the prefix sums,
            t-statistics, the warp-chunked detector for runtime parameters, sequential-order emitter)
  custom    a set of neither reference, (4, 9, 3.0, 1.5, 0.5): the general route with a long detector that emits
Each is timed with CUDA events over --iters runs after --warmup runs; the stage times (SGPU_F_STAGE_TIMERS) come from
one extra run. Every line records the reads summed in the reference's order and the detector chunks redone
(fixups: warm-up states that did not match), and dna_set whether its events equal the default's bit for bit.

Live: tools/live_time.py's device configurations (int16 and pA entries; 512, 3,000 and 144,000 channels) and its host
submit -> wait latency, each without a set and with the custom set, alternated.

Prints one JSON line per configuration, and the card's name, power limit and max SM clock.

    python tools/detector_time.py [--iters 20] [--warmup 3] [--no-live] [--out detector_time.jsonl]
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

CUSTOM = sg.Detector(4, 9, 3.0, 1.5, 0.5)
CONFIGS = {"default": None, "dna_set": sg.Detector(3, 6, 1.4, 9.0, 0.2), "custom": CUSTOM}


def batches(a, dev):
    lens = synth.read_lengths(bench.N_SET)[:a.reads]
    b = bench.device_batch(torch, dev, lens, 0, synth.SEED, 0.1)
    span, n = b["span"], b["n_reads"]
    lines = []
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS) as c, \
            sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS) as ct:
        stream = torch.cuda.current_stream()
        st = stream.cuda_stream

        def run(ctx, det):
            ctx.set_detector(det)
            return ctx.run_device(b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(),
                                  b["offset"].data_ptr(), b["unit"].data_ptr(), n, span, 0, sg.WANT_EVENTS, st)

        out = {}
        for name, det in CONFIGS.items():  # outputs and counters of one run of each
            d = run(c, det)
            torch.cuda.synchronize()
            cnt = c.counters()
            assert cnt["status"] == 0, (name, cnt)
            ne = cnt["n_events"]
            out[name] = {"events": (c.d2h(d.ev_off, np.uint64, n + 1), c.d2h(d.ev_start, np.uint32, ne),
                                    c.d2h(d.ev_mean, np.float32, ne).view(np.uint32),
                                    c.d2h(d.ev_stdv, np.float32, ne).view(np.uint32)),
                         "n_events": ne, "seq_order_reads": int(c.d2h(d.seq_order, np.uint32, n).sum()),
                         "fixup_chunks": int(c.d2h(d.fixups, np.uint32, n).sum()),
                         "launches": cnt["n_kernel_launches"]}
            run(ct, det)
            out[name]["stages"] = [(s, round(ms, 4), k) for s, ms, k in ct.stage_times()]
        for k in range(a.warmup):
            for det in CONFIGS.values():
                run(c, det)
        torch.cuda.synchronize()
        ms = {name: [] for name in CONFIGS}
        for k in range(a.iters):
            for name, det in CONFIGS.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                run(c, det)
                e1.record(stream)
                ms[name].append((e0, e1))
        torch.cuda.synchronize()
        for name in CONFIGS:
            t = np.array([e0.elapsed_time(e1) for e0, e1 in ms[name]])
            o = out[name]
            line = {"config": f"batch_dna_{name}", "detector": None if CONFIGS[name] is None else list(CONFIGS[name]),
                    "reads": n, "samples": span, "runs_timed": a.iters, "ms_median": float(np.median(t)),
                    "ms_min": float(t.min()), "ms_max": float(t.max()), "gsamples_per_s": span / float(np.median(t)) / 1e6,
                    "n_events": o["n_events"], "seq_order_reads": o["seq_order_reads"],
                    "fixup_chunks": o["fixup_chunks"], "launches": o["launches"], "stages": o["stages"]}
            if name == "dna_set":
                line["events_equal_default"] = all(np.array_equal(x, y) for x, y in
                                                   zip(out["default"]["events"], o["events"]))
            lines.append(line)
            print(json.dumps(line), flush=True)
    return lines


def live(a, dev):
    lines = []
    for pa in (False, True):
        for per_push, rna in ((2000, 0), (1200, 1)):
            for channels in (512, 3000, 144000):
                for det in (None, CUSTOM):
                    line = live_time.device_config(dev, channels, per_push, rna, a.iters, a.warmup, pa, det)
                    line["detector"] = None if det is None else list(det)
                    lines.append(line)
                    print(json.dumps(line), flush=True)
        for det in (None, CUSTOM):
            line = live_time.host_latency(3000, 2000, a.iters, a.warmup, pa, det)
            line["detector"] = None if det is None else list(det)
            lines.append(line)
            print(json.dumps(line), flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-live", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lines = [{"card": live_time.card()}]
    print(json.dumps(lines[0]), flush=True)
    lines += batches(a, dev)
    if not a.no_live:
        lines += live(a, dev)
    if a.out:
        with open(a.out, "w") as f:
            for ln_ in lines:
                f.write(json.dumps(ln_) + "\n")


if __name__ == "__main__":
    main()

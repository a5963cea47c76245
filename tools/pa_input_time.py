"""Device-resident throughput of event detection on pA floats (sgpu_run_device_pa), DNA and RNA.

The batch is bench.py's: the first 16,384 reads of the named synthetic set, generated on the GPU (DNA level changes
with p = 0.1, RNA with 0.025). Its pA is produced once by the library itself (an int16 run with SGPU_WANT_PA) and read
before timing. Each configuration is timed with CUDA events over --iters runs after --warmup runs; the per-stage times
(SGPU_F_STAGE_TIMERS) come from one extra run. The same batch runs with every read summed in the reference's order
(SGPU_F_FORCE_GENERIC) for comparison. Prints one JSON line per configuration, and the card's name and power limit.

    python tools/pa_input_time.py [--iters 20] [--warmup 3] [--out pa_input_time.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lens = synth.read_lengths(bench.N_SET)[:a.reads]
    lines = []
    for rna in (0, 1):
        b = bench.device_batch(torch, dev, lens, 0, synth.SEED, 0.025 if rna else 0.1)
        span, n = b["span"], b["n_reads"]
        cap = span + 64
        flags_all = {"scan": sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS,
                     "forced_reference_order": sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS | sg.F_FORCE_GENERIC}
        pa = torch.empty(span, dtype=torch.float32, device=dev)
        with sg.Context(device=0, max_samples=cap, max_reads=n, flags=sg.F_NO_HOST_SLOTS) as c:
            st = torch.cuda.current_stream().cuda_stream
            d = c.run_device(b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(),
                             b["offset"].data_ptr(), b["unit"].data_ptr(), n, span, rna, sg.WANT_EVENTS | sg.WANT_PA, st)
            torch.cuda.synchronize()
            ne16 = c.counters()["n_events"]
            ev16 = c.d2h(d.ev_start, np.uint32, ne16)
            # the library's own pA (through the host: the context's outputs are reused by its next run)
            pa.copy_(torch.from_numpy(c.d2h(d.pa, np.float32, span)).to(dev))
            torch.cuda.synchronize()
        for name, flags in flags_all.items():
            with sg.Context(device=0, max_samples=cap, max_reads=n, flags=flags) as c:
                st = torch.cuda.current_stream().cuda_stream

                def run():
                    return c.run_device_pa(pa.data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr(), n, span,
                                           rna, sg.WANT_EVENTS, st)
                for _ in range(a.warmup):
                    run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    run()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / a.iters
                d = run()
                torch.cuda.synchronize()
                stages = [(s, round(t, 4), k) for s, t, k in c.stage_times()]
                cnt = c.counters()
                same = cnt["n_events"] == ne16 and np.array_equal(c.d2h(d.ev_start, np.uint32, ne16), ev16)
            line = {"tool": "pa_input_time", "rna": rna, "path": name, "reads": n, "samples": int(b["n_samples"]),
                    "ms": round(ms, 4), "gsamples_per_s": round(b["n_samples"] / ms / 1e6, 2),
                    "n_seq_order_reads": cnt["n_seq_order_reads"], "events": cnt["n_events"],
                    "same_events_as_int16_path": bool(same), "stages": stages, "card": card()}
            print(json.dumps(line), flush=True)
            lines.append(line)
        del b
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

"""Device-resident throughput of the statistics of pA records (sgpu_run_device_pa with SGPU_WANT_STAT), in three forms of
one batch, each in both roles of the moments kernel and with the default split:

  pa         the pA the int16 route produces (an int16 run with SGPU_WANT_PA): positive values
  normalised the same pA normalised per read by its median and MAD, (x - median) / MAD: values of either sign, which the
             signed summaries of float_order.cuh take; if this form is far slower than `pa`, they are not engaging
  int16      SGPU_WANT_STAT on the int16 reads themselves (sgpu_run_device), the yardstick

The batch is bench.py's: the first 16,384 reads of the synthetic DNA set, generated on the GPU. The per-read medians
and MADs come from the library's own pA statistics. Before timing, `pa`'s columns 1, 3, 5 are compared bit for bit
with the int16 run's, and 64 reads of `normalised` with sequential float32 loops in numpy. Each configuration is timed
with CUDA events over --iters runs after --warmup runs; the stage times (SGPU_F_STAGE_TIMERS) come from one extra run.
Prints one JSON line per configuration, with the card's name and power limit.

    python tools/pa_stat_time.py [--iters 20] [--warmup 3] [--out pa_stat_time.jsonl]
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
import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import _lib as _sl, synth  # noqa: E402
from pa_input_time import card  # noqa: E402

ROLES = {"cta": 0, "default": 131072, "warp": 1 << 31}


def seq_stat(x):
    """meanf, stdvf, medianf in float32, summed one value after the other"""
    x = np.asarray(x, np.float32)
    n = np.float32(len(x))
    zero = np.zeros(1, np.float32)                     # the loops start from +0
    m = np.add.accumulate(np.concatenate([zero, x]), dtype=np.float32)[-1] / n
    d = x - m
    s = np.sqrt(np.add.accumulate(np.concatenate([zero, d * d]), dtype=np.float32)[-1] / n)
    return np.array([m, s, np.sort(x)[len(x) // 2]], np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lens = synth.read_lengths(bench.N_SET)[:a.reads]
    b = bench.device_batch(torch, dev, lens, 0, synth.SEED, 0.1)
    span, n = b["span"], b["n_reads"]
    off, ln = b["read_off"], b["read_len"]
    flags = sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS | sg.F_PA_STAT
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=flags) as c:
        st = torch.cuda.current_stream().cuda_stream

        def int16(want):
            return c.run_device(b["samples"].data_ptr(), off.data_ptr(), ln.data_ptr(), b["offset"].data_ptr(),
                                b["unit"].data_ptr(), n, span, 0, want, st)

        def pa_stat(x):
            d = c.run_device_pa(x.data_ptr(), off.data_ptr(), ln.data_ptr(), n, span, 0, sg.WANT_STAT, st)
            torch.cuda.synchronize()
            return c.d2h(d.stat, np.float32, 6 * n).reshape(n, 6)

        d = int16(sg.WANT_PA | sg.WANT_STAT)
        torch.cuda.synchronize()
        stat16 = c.d2h(d.stat, np.float32, 6 * n).reshape(n, 6)
        pa = torch.from_numpy(c.d2h(d.pa, np.float32, span)).to(dev)   # (the context's outputs are reused)
        st_pa = pa_stat(pa)
        same_pa = bool(np.array_equal(st_pa[:, [1, 3, 5]].view(np.uint32), stat16[:, [1, 3, 5]].view(np.uint32)))
        # median / MAD normalisation on the device, from the library's own medians
        lens_al = (off[1:] - off[:-1])
        med = torch.repeat_interleave(torch.from_numpy(st_pa[:, 5].copy()).to(dev), lens_al, output_size=span)
        dev_abs = (pa - med).abs()
        mad = torch.repeat_interleave(torch.from_numpy(pa_stat(dev_abs)[:, 5].copy()).to(dev), lens_al,
                                      output_size=span).clamp_min(1e-3)
        norm = (pa - med) / mad
        del dev_abs, med, mad
        st_norm = pa_stat(norm)
        rng = np.random.default_rng(1)
        flat = norm.cpu().numpy()
        offs, lns = off.cpu().numpy(), ln.cpu().numpy()
        checked = [int(r) for r in rng.choice(n, 64, replace=False)]
        same_norm = all(np.array_equal(seq_stat(flat[offs[r]:offs[r] + lns[r]]).view(np.uint32),
                                       st_norm[r, [1, 3, 5]].view(np.uint32)) for r in checked if lns[r])
        negative_share = float((flat < 0).sum()) / float(lns.sum())
        del flat
        lines = []
        forms = {"pa": lambda: c.run_device_pa(pa.data_ptr(), off.data_ptr(), ln.data_ptr(), n, span, 0,
                                               sg.WANT_STAT, st),
                 "normalised": lambda: c.run_device_pa(norm.data_ptr(), off.data_ptr(), ln.data_ptr(), n, span, 0,
                                                       sg.WANT_STAT, st),
                 "int16": lambda: int16(sg.WANT_STAT)}
        for role, cta_min in ROLES.items():
            c.set_param(_sl.PARAM_STAT_CTA_MIN, cta_min)
            for form, run in forms.items():
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
                run()
                torch.cuda.synchronize()
                stages = [(s, round(t, 4), k) for s, t, k in c.stage_times()]
                line = {"tool": "pa_stat_time", "form": form, "role": role, "stat_cta_min": cta_min, "reads": n,
                        "samples": int(b["n_samples"]), "ms": round(ms, 4),
                        "gsamples_per_s": round(b["n_samples"] / ms / 1e6, 2), "stages": stages,
                        "launches": c.counters()["n_kernel_launches"], "card": card()}
                if form == "pa":
                    line["same_as_int16_route"] = same_pa
                if form == "normalised":
                    line["same_as_sequential_loops_on_64_reads"] = bool(same_norm)
                    line["negative_share"] = round(negative_share, 4)
                print(json.dumps(line), flush=True)
                lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()

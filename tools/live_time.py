"""Device time of live pushes (sgpu_run_device_live, and sgpu_run_device_live_pa for entries of pA floats): every
channel gets one entry of P samples per push, and every push continues the reads of the previous one (the first opens
them).

Configurations: 512, 3,000 and 144,000 channels (a MinION, a GridION-sized load, a full PromethION) with 2,000
samples per push (DNA: 0.4 s at 5 kHz) and with 1,200 (RNA: 0.4 s at 3 kHz); and the host path's submit -> wait
latency of one push of the 3,000-channel DNA case (sgpu_submit + sgpu_wait_live, the slot filled beforehand).
The signal is generated on the GPU (a level per 10 samples, uniform noise); the pA entries are the same samples
calibrated to floats. NBUF different pushes are cycled. Each device configuration is timed with CUDA events around
every push over --iters pushes after --warmup. --input picks the int16 configurations, the pA ones (named *_pa_*) or
both. Prints one JSON line per configuration, and the card's name, power limit and max SM clock.

    python tools/live_time.py [--iters 20] [--warmup 3] [--input int16|pa|both] [--out live_time.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import _lib, synth  # noqa: E402

NBUF = 4


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def signal(dev, n, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    lvl = torch.randint(300, 700, (n // 10 + 1,), device=dev, generator=g).repeat_interleave(10)[:n]
    return (lvl + torch.randint(-20, 21, (n,), device=dev, generator=g)).to(torch.int16)


def device_config(dev, channels, per_push, rna, iters, warmup, pa=False, det=None):
    """det: a detector set (sgpu_set_detector) in force for the pushes, or None: the reference's"""
    n = channels * per_push
    unit = np.float32(synth.RANGE) / np.float32(synth.DIGITISATION)
    bufs = [signal(dev, n, 100 + k) for k in range(NBUF)]
    if pa:  # misc.c:28 with offset 0: the pA the int16 entries stand for
        bufs = [b.to(torch.float32) * float(unit) for b in bufs]
    off = torch.arange(channels + 1, device=dev, dtype=torch.int64) * per_push
    ln = torch.full((channels,), per_push, device=dev, dtype=torch.int32)
    ch = torch.arange(channels, device=dev, dtype=torch.int32)
    first = torch.full((channels,), sg.LIVE_START | (sg.LIVE_RNA if rna else 0), device=dev, dtype=torch.int32)
    later = torch.zeros(channels, device=dev, dtype=torch.int32)
    offs = torch.full((channels,), 0.0, device=dev, dtype=torch.float32)
    units = torch.full((channels,), float(unit), device=dev, dtype=torch.float32)
    with sg.Context(device=0, max_samples=n, max_reads=channels, flags=sg.F_NO_HOST_SLOTS) as c:
        c.live_open(channels)
        c.set_detector(det)
        stream = torch.cuda.current_stream()
        st = stream.cuda_stream
        if pa:
            push = lambda k, flags: c.run_device_live_pa(  # noqa: E731
                bufs[k % NBUF].data_ptr(), off.data_ptr(), ln.data_ptr(), ch.data_ptr(), flags.data_ptr(), channels, n, st)
        else:
            push = lambda k, flags: c.run_device_live(  # noqa: E731
                bufs[k % NBUF].data_ptr(), off.data_ptr(), ln.data_ptr(), ch.data_ptr(), flags.data_ptr(), offs.data_ptr(),
                units.data_ptr(), channels, n, st)
        for k in range(warmup):
            push(k, first if k == 0 else later)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for k in range(iters):
            ev[k][0].record(stream)
            push(warmup + k, later)
            ev[k][1].record(stream)
        torch.cuda.synchronize()
        ms = np.array([a.elapsed_time(b) for a, b in ev])
        cnt = c.counters()
        assert cnt["status"] == 0, cnt
    return {"config": f"device_{'pa_' if pa else ''}{'rna' if rna else 'dna'}_{channels}ch", "input": "pa" if pa else "int16",
            "channels": channels, "samples_per_push": per_push,
            "rna": rna, "pushes_timed": iters, "ms_median": float(np.median(ms)), "ms_min": float(ms.min()),
            "ms_max": float(ms.max()), "gsamples_per_s": n / float(np.median(ms)) / 1e6,
            "events_last_push": cnt["n_events"], "launches_per_push": cnt["n_kernel_launches"]}


def host_latency(channels, per_push, iters, warmup, pa=False, det=None):
    raws = np.random.default_rng(7).integers(300, 700, size=(channels, per_push * (warmup + iters))).astype(np.int16)
    unit = np.float32(synth.RANGE) / np.float32(synth.DIGITISATION)
    lib = _lib.load()
    out = []
    # (a slot holds max_samples / 2 floats)
    with sg.Context(device=0, max_samples=channels * per_push * (2 if pa else 1), max_reads=channels, n_slots=1) as c:
        c.live_open(channels)
        c.set_detector(det)
        res = _lib.LiveResult()
        for k in range(warmup + iters):
            flags = sg.LIVE_START if k == 0 else 0
            chunk = lambda q: raws[q][k * per_push:(k + 1) * per_push]  # noqa: E731
            if pa:
                c.live_fill_pa(0, [(q, flags, (chunk(q) + np.float32(q % 53)) * unit) for q in range(channels)])
            else:
                c.live_fill(0, [(q, flags, chunk(q), synth.DIGITISATION, float(q % 53), synth.RANGE)
                                for q in range(channels)])
            t0 = time.perf_counter()
            rc = lib.sgpu_submit(c._h, 0, sg.WANT_EVENTS)
            rc = rc or lib.sgpu_wait_live(c._h, 0, C.byref(res))
            t1 = time.perf_counter()
            assert rc == 0, rc
            if k >= warmup:
                out.append((t1 - t0) * 1e3)
    ms = np.array(out)
    return {"config": f"host_{'pa_' if pa else ''}dna_{channels}ch_submit_to_wait", "input": "pa" if pa else "int16",
            "channels": channels, "samples_per_push": per_push,
            "pushes_timed": iters, "ms_median": float(np.median(ms)), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
            "events_last_push": int(res.n_events)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--input", choices=("int16", "pa", "both"), default="int16")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    forms = {"int16": (False,), "pa": (True,), "both": (False, True)}[a.input]
    dev = torch.device("cuda:0")
    lines = [{"card": card()}]
    print(json.dumps(lines[0]), flush=True)
    for pa in forms:
        for per_push, rna in ((2000, 0), (1200, 1)):
            for channels in (512, 3000, 144000):
                lines.append(device_config(dev, channels, per_push, rna, a.iters, a.warmup, pa))
                print(json.dumps(lines[-1]), flush=True)
        lines.append(host_latency(3000, 2000, a.iters, a.warmup, pa))
        print(json.dumps(lines[-1]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for ln_ in lines:
                f.write(json.dumps(ln_) + "\n")


if __name__ == "__main__":
    main()

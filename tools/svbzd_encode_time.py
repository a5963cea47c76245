"""Device time of the svb-zd encoder (sgpu_encode_svbzd_device, SGPU_WANT_SVBZD) next to the decoder.

Batches, device resident (int16 samples generated on the GPU by bench.device_batch):
  bench  bench.py's synthetic DNA batch: the first 16,384 reads of its set
  long   320 reads of 2,000,000 samples of the same generator
Per batch, after --warmup runs of each, --iters rounds alternate one encode (sgpu_encode_svbzd_device) and one decode
of its output (sgpu_decode_svbzd_device, the output fed in unchanged), each timed with CUDA events on the stream it runs
on. Both working sets exceed the 126 MB L2. Before timing, the decode of the encoder's output is checked to give the
batch's samples back, and the first 64 streams to equal sigtk_b200.synth.svbzd_encode.

Host slots: the first --host-reads reads of the bench batch through one pinned slot (fill once, then submit + wait),
SGPU_WANT_EVENTS with and without SGPU_WANT_SVBZD alternated, timed with the host clock around sgpu_submit, sgpu_wait
and sgpu_slot_svbzd (copies included; the unpacking into numpy arrays excluded).

Each line gives Gsamples/s (median over the rounds), the stream bytes per sample (sum of comp_len, and comp_off[n]
with the padding to 16 bytes), and the card's name, power limit and max SM clock read in the same call.

    python tools/svbzd_encode_time.py [--iters 20] [--warmup 3] [--host-reads 4096] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import live_time  # noqa: E402
import sigtk_b200 as sg  # noqa: E402
from sigtk_b200 import synth  # noqa: E402


def timed(fn, st):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b)


def time_device(name, b, a, card):
    n, span, n_samp = b["n_reads"], b["span"], b["n_samples"]
    lens = b["host_len"]
    n_blocks = int(((lens + 1023) // 1024).sum())
    st = torch.cuda.current_stream()
    with sg.Context(device=0, max_samples=span + 64, max_reads=n, flags=sg.F_NO_HOST_SLOTS) as c:
        out = torch.zeros(span, dtype=torch.int16, device="cuda")
        ptrs = (b["samples"].data_ptr(), b["read_off"].data_ptr(), b["read_len"].data_ptr())

        def enc():
            return c.encode_svbzd_device(*ptrs, n, span, st.cuda_stream)

        res = enc()
        comp_off = c.d2h(res.comp_off, np.uint64, n + 1)
        comp_len = c.d2h(res.comp_len, np.uint32, n)
        n_bytes = int(comp_off[n])

        def dec():
            c.decode_svbzd_device(res.bytes, n_bytes, res.comp_off, res.comp_len, ptrs[1], ptrs[2], n, n_blocks,
                                  out.data_ptr(), st.cuda_stream)

        dec()
        torch.cuda.synchronize()
        assert c.counters()["status"] == 0
        assert torch.equal(out, b["samples"]), "decoded samples differ"  # (padding: zeros in both)
        flat = c.d2h(res.bytes, np.uint8, int(comp_off[64]))
        host = bench.host_reads_of(b, 64)
        for r in range(64):
            s = flat[int(comp_off[r]): int(comp_off[r]) + int(comp_len[r])]
            assert np.array_equal(s, synth.svbzd_encode(host[r][0])), f"stream {r} differs"
        for _ in range(a.warmup):
            enc()
            dec()
        te, td = [], []
        for _ in range(a.iters):
            te.append(timed(enc, st))
            td.append(timed(dec, st))
    lines = []
    for what, ms in (("encode", te), ("decode", td)):
        ms = np.array(ms)
        lines.append({"batch": name, "path": "device", "kernel": what, "reads": n, "samples": n_samp,
                      "runs_timed": a.iters,
                      "ms": {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())},
                      "gsamples_per_s": n_samp / float(np.median(ms)) / 1e6,
                      "stream_bytes_per_sample": float(comp_len.astype(np.int64).sum()) / n_samp,
                      "buffer_bytes_per_sample": n_bytes / n_samp, "checked": "decode == samples, 64 streams == numpy encoder",
                      "card": card})
    return lines


def time_host(b, a, card):
    reads = bench.host_reads_of(b, a.host_reads)
    n_samp = int(sum(len(r[0]) for r in reads))
    span = int(sum((len(r[0]) + 7) // 8 * 8 for r in reads))
    wants = {"events": sg.WANT_EVENTS, "events+svbzd": sg.WANT_EVENTS | sg.WANT_SVBZD}
    with sg.Context(device=0, max_samples=span + 64, max_reads=len(reads), n_slots=1) as c:
        c.fill(0, reads, 0)
        outs = {}
        for k, w in wants.items():
            c.submit(0, w)
            outs[k] = c.wait(0, w)
        res, svb = sg._lib.Result(), sg._lib.SvbResult()
        t = {k: [] for k in wants}
        for it in range(a.warmup + a.iters):
            for k, w in wants.items():
                t0 = time.perf_counter()
                c.submit(0, w)
                c._check(c._lib.sgpu_wait(c._h, 0, C.byref(res)))
                if w & sg.WANT_SVBZD:
                    c._check(c._lib.sgpu_slot_svbzd(c._h, 0, C.byref(svb)))
                if it >= a.warmup:
                    t[k].append(time.perf_counter() - t0)
        ev, both = outs["events"], outs["events+svbzd"]
        assert np.array_equal(ev.ev_start, both.ev_start) and np.array_equal(ev.ev_mean.view(np.uint32),
                                                                              both.ev_mean.view(np.uint32))
        comp = int(sum(len(s) for s in both.svbzd))
    lines = []
    for k in wants:
        s = np.array(t[k])
        line = {"batch": "bench", "path": "host_slot", "want": k, "reads": len(reads), "samples": n_samp,
                "runs_timed": a.iters,
                "ms": {"median": 1e3 * float(np.median(s)), "min": 1e3 * float(s.min()), "max": 1e3 * float(s.max())},
                "gsamples_per_s": n_samp / float(np.median(s)) / 1e9, "card": card}
        if k == "events+svbzd":
            line["stream_bytes_per_sample"] = comp / n_samp
            line["d2h_stream_bytes"] = int(svb.n_bytes)
        lines.append(line)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reads", type=int, default=4096)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    card = live_time.card()
    lines = []
    for name in ("bench", "long"):
        lens = synth.read_lengths(bench.N_SET)[:16384] if name == "bench" else np.full(320, 2_000_000, np.int64)
        b = bench.device_batch(torch, dev, lens, 0, synth.SEED, 0.1)
        torch.cuda.synchronize()
        new = time_device(name, b, a, card)
        if name == "bench":
            new += time_host(b, a, card)
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

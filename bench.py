#!/usr/bin/env python
"""bench.py -- event-detection throughput of the sigtk B200 hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--reads-per-step B] [--mode event+pa|event]
                  [--dump-outputs DIR]

A "step" = one pass of the hot path (pA conversion + event detection, event table out, pA materialised in the
default `event+pa` mode) over one device-resident batch of B synthetic DNA reads drawn from the 1,000,000-read
set of BASELINE.json configs[2] (int16, lognormal length, mean 40,000 samples, sigma 0.6; SURVEY.md 8(d)).
Reads are independent, so with N GPUs every rank processes its own batches (weak scaling, no collective on the
data path; torch.distributed is used for the barrier and the max-over-ranks only).

  value      whole-job Gsamples/s, inputs resident in HBM, CUDA-event time of the K steps, max over ranks
  e2e        the same metric through the host C-ABI (pinned slot -> sgpu_submit -> sgpu_wait): H2D of the samples
             and D2H of the event table (+ pA in event+pa mode) inside the timed region
  roofline   dominant kernel (walk_chunks_kernel): algorithmic bytes of the path per launch / its CUDA-event time
  cpu_baseline  the UNMODIFIED reference functions (oracle/_ref/libsigtk_ref.so: signal_in_picoamps + getevents)
             on 1 host thread over a bounded sample of the same reads (N=1, rank 0 only)

--impl reference times the reference's CPU path on all host threads (one reference call chain per thread over
disjoint reads) and prints the same line with "impl": "reference".

--dump-outputs DIR writes what the last timed step returned (rank 0) as .npy files, so that two builds can be compared
output for output on the same inputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from sigtk_b200 import synth  # noqa: E402

N_SET = 1_000_000          # reads of the named synthetic set
METRIC = "event_detection_throughput"
UNIT = "Gsamples/s"
WORKLOAD = "synthetic 1M DNA reads, int16, lognormal length mean 40k samples (sigma 0.6), {mode}"
WORKLOADS = {"dna40k": WORKLOAD,
             "dna178k": "synthetic DNA reads, int16, fixed 178,000 samples (20 kb-equivalent), {mode}",
             "ultralong": "synthetic ultra-long DNA reads, int16, 2,000,000 samples each, {mode}",
             "rna40k": "synthetic RNA-parameter reads, int16, lognormal length mean 40k samples, {mode}",
             "real": "the 100 R9.4 DNA reads of test/sp1_dna.blow5 (tests/golden/sp1_dna.npz) tiled to >= 300 M samples, {mode}"}


def alg_bytes(n_samples: int, n_reads: int, n_events: int, pa: bool) -> int:
    """SURVEY.md 8(d) / BASELINE.md 4: algorithmic bytes of the path."""
    return 2 * n_samples + 20 * n_reads + 12 * n_events + 8 * n_reads + (4 * n_samples if pa else 0)


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.rows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
def pin_to_gpu_numa(torch, local: int, world: int) -> dict:
    """Run this rank on the cores of the NUMA node its GPU hangs off (pinned host buffers are then allocated there:
    first touch), the node's cores shared evenly by the ranks on it. The end-to-end number is a PCIe number; a DMA
    that crosses the socket interconnect runs at a fraction of the link rate."""
    info = {"numa_node": None, "cpus": None}
    try:
        pr = torch.cuda.get_device_properties(local)
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return info
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return info
        # ranks whose GPUs share this node split its cores
        peers = []
        for g in range(world):
            q = torch.cuda.get_device_properties(g)
            b2 = f"{q.pci_domain_id:04x}:{q.pci_bus_id:02x}:{q.pci_device_id:02x}.0"
            try:
                if int(open(f"/sys/bus/pci/devices/{b2}/numa_node").read().strip()) == node:
                    peers.append(g)
            except Exception:
                pass
        k, m = peers.index(local) if local in peers else 0, max(len(peers), 1)
        share = allowed[k * len(allowed) // m:(k + 1) * len(allowed) // m] or allowed
        os.sched_setaffinity(0, share)
        info = {"numa_node": node, "cpus": f"{share[0]}-{share[-1]} ({len(share)})"}
    except Exception as e:  # no sysfs / no permission: run unpinned
        info["error"] = str(e)[:80]
    return info


def copy_only_ceiling(torch, dev, h2d_bytes: int, d2h_bytes: int, steps: int, dist):
    """The PCIe ceiling of the end-to-end path: the same bytes per step as run_e2e moves, pinned host memory, H2D
    and D2H on two streams at once, NO kernels. seconds (max over ranks) for `steps` steps."""
    hin = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    hout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    din = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=dev)
    dout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    for _ in range(2):
        with torch.cuda.stream(s_in):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s_out):
            hout.copy_(dout, non_blocking=True)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        with torch.cuda.stream(s_in):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s_out):
            hout.copy_(dout, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _mix_t(torch, x):
    """splitmix64 finaliser on int64 tensors (two's-complement wrap-around = uint64 arithmetic; logical shifts by masking)"""
    def c(v):
        return v - (1 << 64) if v >= (1 << 63) else v
    x = x ^ ((x >> 30) & ((1 << 34) - 1))
    x = x * c(synth._M1)
    x = x ^ ((x >> 27) & ((1 << 37) - 1))
    x = x * c(synth._M2)
    x = x ^ ((x >> 31) & ((1 << 33) - 1))
    return x


def device_batch(torch, dev, lens: np.ndarray, first_index: int, seed: int, p_change: float = 0.1):
    """One batch of the counter-based synthetic set generated on the device: read k of the batch is read
    first_index + k of the named set, bit-identical to sigtk_b200.synth.make_read_cb (same integer hashes, same exactly
    rounded float64 operations; tests/test_synth.py) whatever the device, rank or batch boundaries.
    -> dict(samples i16[span], read_off i64[n+1], read_len i32[n], offset f32[n], unit f32[n], span, n_samples)"""
    def c(v):
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v
    n = len(lens)
    al = (lens + 7) // 8 * 8
    off = np.zeros(n + 1, dtype=np.int64)
    off[1:] = np.cumsum(al)
    span = int(off[-1])
    samples = torch.zeros(span, dtype=torch.int16, device=dev)
    index = first_index + np.arange(n, dtype=np.int64)
    offsets = (index % 53).astype(np.float32)
    keys = synth.read_key(seed, index).view(np.int64)
    scale = synth.DIGITISATION / synth.RANGE
    thr = int(p_change * (1 << 24))
    CH = 1 << 24
    r0 = 0
    while r0 < n:  # groups of whole reads of about CH samples
        r1 = int(np.searchsorted(off, off[r0] + CH, side="right"))
        r1 = min(max(r1 - 1, r0 + 1), n)
        a, b = int(off[r0]), int(off[r1])
        m = b - a
        reps = torch.from_numpy(al[r0:r1]).to(dev)
        key = torch.repeat_interleave(torch.from_numpy(keys[r0:r1]).to(dev), reps, output_size=m)
        rstart = torch.repeat_interleave(torch.from_numpy(off[r0:r1] - a).to(dev), reps, output_size=m)
        pos = torch.arange(m, dtype=torch.int64, device=dev)
        i = pos - rstart                                      # sample index inside its read (padding included)

        def h(ii, stream):
            return _mix_t(torch, key ^ (ii * c(synth._K_SAMPLE) + c(stream * synth._K_STREAM)))

        change = ((h(i, 1) >> 40) & ((1 << 24) - 1)) < thr
        change |= i == 0
        start = torch.cummax(torch.where(change, pos, torch.full_like(pos, -1)), 0).values - rstart
        del change
        u = ((h(start, 2) >> 11) & ((1 << 53) - 1)).to(torch.float64) * (1.0 / 9007199254740992.0)
        pa = 60.0 + 60.0 * u
        del u, start
        tot = torch.zeros(m, dtype=torch.int64, device=dev)
        for s in (3, 4, 5):
            hh = h(i, s)
            for k in range(4):
                tot += (hh >> (16 * k)) & 0xFFFF
            del hh
        pa += (tot - 393210).to(torch.float64) * (2.0 / 65536.0)
        del tot
        o = torch.repeat_interleave(torch.from_numpy(offsets[r0:r1].astype(np.float64)).to(dev), reps, output_size=m)
        raw = torch.round(pa * scale - o).clamp_(-32768, 32767).to(torch.int16)
        ln = torch.repeat_interleave(torch.from_numpy(lens[r0:r1]).to(dev), reps, output_size=m)
        raw[i >= ln] = 0                                      # the padding up to the next multiple of 8 samples
        samples[a:b] = raw
        del pa, o, raw, key, rstart, pos, i, ln
        r0 = r1
    unit = (np.float32(synth.RANGE) / np.float32(synth.DIGITISATION)).astype(np.float32)
    return {
        "samples": samples,
        "read_off": torch.from_numpy(off).to(dev),
        "read_len": torch.from_numpy(lens.astype(np.int32)).to(dev),
        "offset": torch.from_numpy(offsets).to(dev),
        "unit": torch.full((n,), float(unit), dtype=torch.float32, device=dev),
        "span": span, "n_samples": int(lens.sum()), "n_reads": n, "host_off": off, "host_len": lens,
        "host_offset": offsets,
    }


def host_reads_of(batch, n_first: int):
    """first reads of a device batch as the (raw, digitisation, offset, range) tuples the checkers take"""
    off, lens = batch["host_off"], batch["host_len"]
    n_first = min(n_first, len(lens))
    flat = batch["samples"][: int(off[n_first])].cpu().numpy()
    dig, rng = batch.get("host_dig"), batch.get("host_range")
    return [(flat[int(off[r]): int(off[r]) + int(lens[r])].copy(), synth.DIGITISATION if dig is None else float(dig[r]),
             float(batch["host_offset"][r]), synth.RANGE if rng is None else float(rng[r])) for r in range(n_first)]


def real_batch(torch, dev, target_samples: int = 300_000_000):
    """The reference's own fixture (100 real R9.4 reads, 472,511 samples) repeated until the batch holds
    target_samples: real glitches, stalls and reads whose sums are order dependent (1 in 100 fails the exact-sum
    witness and takes the sequential-order kernels) -- what the synthetic model does not have."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "sp1_dna.npz"), allow_pickle=True)
    roff = z["read_off"].astype(np.int64)
    lens1 = np.diff(roff)
    copies = int(-(-target_samples // int(lens1.sum())))
    lens = np.tile(lens1, copies)
    n = len(lens)
    al = (lens + 7) // 8 * 8
    off = np.zeros(n + 1, dtype=np.int64)
    off[1:] = np.cumsum(al)
    one = np.zeros(int(al[:len(lens1)].sum()), dtype=np.int16)
    for r in range(len(lens1)):
        one[int(off[r]): int(off[r]) + int(lens1[r])] = z["samples"][int(roff[r]): int(roff[r + 1])]
    samples = torch.from_numpy(one).to(dev).repeat(copies)
    offsets = np.tile(z["offset"].astype(np.float32), copies)
    unit1 = (z["range"].astype(np.float32) / z["digitisation"].astype(np.float32)).astype(np.float32)  # misc.c:17-19,26
    unit = np.tile(unit1, copies)
    return {
        "samples": samples, "read_off": torch.from_numpy(off).to(dev), "read_len": torch.from_numpy(lens.astype(np.int32)).to(dev),
        "offset": torch.from_numpy(offsets).to(dev), "unit": torch.from_numpy(unit).to(dev),
        "span": int(off[-1]), "n_samples": int(lens.sum()), "n_reads": n, "host_off": off, "host_len": lens,
        "host_offset": offsets, "copies": copies,
        "host_dig": np.tile(z["digitisation"], copies), "host_range": np.tile(z["range"], copies),
    }


def short_run(torch, sg, local, batches, rna, want, steps=3, warmup=3):
    """a short device-resident timing of one workload (the extra sub-lines of the default bench line):
    -> dict(value Gsamples/s, ms_per_step, stage ms, counters of the last step)"""
    max_span = max(p["span"] for p in batches)
    max_reads = max(p["n_reads"] for p in batches)
    ctx = sg.Context(device=local, max_samples=max_span, max_reads=max_reads, flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS)
    stream = torch.cuda.current_stream().cuda_stream

    def step(p):
        ctx.run_device(p["samples"].data_ptr(), p["read_off"].data_ptr(), p["read_len"].data_ptr(), p["offset"].data_ptr(),
                       p["unit"].data_ptr(), p["n_reads"], p["span"], rna, want, stream)

    for w in range(warmup):
        step(batches[w % len(batches)])
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = {}
    ns = 0
    ev0.record()
    for k in range(steps):
        p = batches[(warmup + k) % len(batches)]
        step(p)
        ns += p["n_samples"]
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    for k in range(steps):               # per-kernel times: the same steps again (see main)
        step(batches[(warmup + k) % len(batches)])
        for name, ms_, _ in ctx.stage_times():
            stage_ms[name] = stage_ms.get(name, 0.0) + ms_
    c = ctx.counters()
    ctx.close()
    last = batches[(warmup + steps - 1) % len(batches)]
    return {"value": ns / (ms * 1e-3) / 1e9, "unit": UNIT, "steps": steps, "ms_per_step": ms / steps,
            "samples_per_step": ns // steps, "reads_per_step": last["n_reads"],
            "stage_ms_per_step": {k: round(v / steps, 4) for k, v in stage_ms.items()},
            "sequential_order_reads": c["n_seq_order_reads"], "detector_fixups": c["n_fixups"],
            "long_detector_replays": c["n_long_jobs"], "events_per_sample": c["n_events"] / max(last["n_samples"], 1),
            "status": c["status"]}


# ---------------------------------------------------------------------------------------------------------------
def load_checker():
    """the CPU arm: the compiled, unmodified reference if present, else the oracle port"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    if _oracle.have_ref():
        return _oracle.Reference(), "reference"
    return _oracle.Oracle(), "port"


def cpu_time_reads(chk, reads, threads: int):
    """seconds (wall) for pA + event detection of `reads` on `threads` host threads; -> (seconds, samples, events)"""
    if threads <= 1:
        return chk.time_events(reads, 0)
    shards = [reads[k::threads] for k in range(threads)]
    shards = [s for s in shards if s]
    out = [None] * len(shards)

    def work(k):
        out[k] = chk.time_events(shards[k], 0)  # ctypes releases the GIL during the call

    th = [threading.Thread(target=work, args=(k,)) for k in range(len(shards))]
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    return dt, sum(o[1] for o in out), sum(o[2] for o in out)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    chk, kind = load_checker()
    threads = os.cpu_count() or 1
    per_thread = 24
    lens = synth.read_lengths(N_SET)
    reads_per_step = threads * per_thread
    pool = []
    for j in range(3):  # three distinct samples, cycled
        base = j * reads_per_step
        pool.append([synth.make_read_cb(base + i, int(lens[base + i])) for i in range(reads_per_step)])
    for w in range(args.warmup):
        cpu_time_reads(chk, pool[w % 3], threads)
    t_tot, s_tot, e_tot = 0.0, 0, 0
    for k in range(args.steps):
        dt, ns, ne = cpu_time_reads(chk, pool[k % 3], threads)
        t_tot += dt; s_tot += ns; e_tot += ne
    val = s_tot / t_tot / 1e9
    sample = f"{reads_per_step} reads (~{s_tot // max(args.steps, 1)} samples) per step, first reads of the set"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(mode=args.mode), "reads_per_step": reads_per_step},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import sigtk_b200 as sg

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sigtk_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_to_gpu_numa(torch, local, world) if not args.no_affinity else {"numa_node": None, "cpus": "unpinned"}
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod
    pa_mode = args.mode == "event+pa"
    want = sg.WANT_EVENTS | (sg.WANT_PA if pa_mode else 0)
    B = args.reads_per_step
    rna = 1 if args.workload == "rna40k" else 0
    p_change = 0.025 if rna else 0.1
    if args.workload == "dna178k":      # SURVEY 8(d) C3': "20 kb-equivalent" reads, fixed 178,000 samples
        lens_all = np.full(N_SET, 178_000, dtype=np.int64)
        B = min(B, 3670)
    elif args.workload == "ultralong":  # BASELINE config 5: 2,000,000-sample reads
        lens_all = np.full(N_SET, 2_000_000, dtype=np.int64)
        B = min(B, 320)
    else:
        lens_all = synth.read_lengths(N_SET, sigma=args.len_sigma) if args.len_sigma else synth.read_lengths(N_SET)
    if args.fixed_len:                  # development: every read the same length
        lens_all = np.full(N_SET, args.fixed_len, dtype=np.int64)
    pool_n = max(1, min(args.pool, args.steps + args.warmup))
    from sigtk_b200.shard import shard_ranges
    pool = []
    if args.workload == "real":
        pool_n = 1
        pool.append(real_batch(torch, dev))
    for j in range(pool_n if args.workload != "real" else 0):
        # step j works on the next world*B reads of the set, split into contiguous read ranges balanced by samples
        g0 = (j * world * B) % (N_SET - world * B)
        lo, hi = shard_ranges(lens_all[g0:g0 + world * B], world)[rank]
        pool.append(device_batch(torch, dev, lens_all[g0 + lo:g0 + hi], g0 + lo, synth.SEED, p_change))
    torch.cuda.synchronize()
    max_span = max(p["span"] for p in pool)
    max_reads = max(p["n_reads"] for p in pool)
    ctx = sg.Context(device=local, max_samples=max_span, max_reads=max_reads,
                     flags=sg.F_NO_HOST_SLOTS | sg.F_STAGE_TIMERS)
    if args.chunk_len:      # development: SGPU_PARAM_CHUNK_LEN / _WARMUP (never change results; 0 = automatic)
        ctx.set_param(sg._lib.PARAM_CHUNK_LEN, args.chunk_len)
    if args.detector_warmup:
        ctx.set_param(sg._lib.PARAM_WARMUP, args.detector_warmup)
    stream = torch.cuda.current_stream().cuda_stream

    def step(p):
        return ctx.run_device(p["samples"].data_ptr(), p["read_off"].data_ptr(), p["read_len"].data_ptr(),
                              p["offset"].data_ptr(), p["unit"].data_ptr(), p["n_reads"], p["span"], rna, want, stream)

    for w in range(args.warmup):
        step(pool[w % pool_n])
    torch.cuda.synchronize()
    c0 = ctx.counters()
    if c0["status"] != 0:
        raise SystemExit(f"bench.py: device status {c0['status']}")
    if dist:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms, stage_launches = {}, {}
    n_samples = n_events = n_reads = launches = 0
    B_step = sum(p["n_reads"] for p in pool) // len(pool)
    torch.cuda.synchronize()
    ev0.record()
    last = None
    for k in range(args.steps):          # the timed region: K steps launched back to back, no host synchronisation
        p = pool[(args.warmup + k) % pool_n]
        last = (p, step(p))
        n_samples += p["n_samples"]
        n_reads += p["n_reads"]
    ev1.record()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    ms_total = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0 and last is not None:  # before the next run overwrites the result buffers
        dump_outputs(ctx, *last, pa_mode, args.dump_outputs)
    # per-kernel times: the same K steps once more, the stage events (CUDA events on the launch stream) read after
    # every step. Reading them inside the timed region costs a host synchronisation per step: 1 % of the step with one
    # rank on the box, 8 % with eight (r02: 5.61 ms against 5.18).
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    for k in range(args.steps):
        step(pool[(args.warmup + k) % pool_n])
        for name, ms, nl in ctx.stage_times():  # waits for this step's last kernel
            stage_ms[name] = stage_ms.get(name, 0.0) + ms
            stage_launches[name] = nl
    ev3.record()
    torch.cuda.synchronize()
    ms_instrumented = ev2.elapsed_time(ev3)
    clocks = sampler.stop() if rank == 0 else None
    # events per step (counters of the last run x steps would be wrong for a pool of different batches)
    ev_per_batch = []
    for p in pool:
        step(p)
        torch.cuda.synchronize()
        c = ctx.counters()
        ev_per_batch.append((c["n_events"], c["n_seq_order_reads"], c["n_fixups"], c["n_kernel_launches"], c["status"],
                             c["n_long_jobs"]))
    for k in range(args.steps):
        e = ev_per_batch[(args.warmup + k) % pool_n]
        n_events += e[0]
        launches += e[3]
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(n_samples), float(n_events), float(n_reads)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max = float(t.item())
    all_samples, all_events, all_reads = (float(x) for x in tot.tolist())
    value = all_samples / (ms_max * 1e-3) / 1e9

    # ---- the siblings of the event path (`sigtk pa`, `sigtk stat`, `sigtk ent`, `sigtk jnn`, `sigtk prefix`), device resident, on the first batch ----------------
    siblings = {}
    if not args.no_siblings:
        p0 = pool[0]
        for name, w_ in (("pa", sg.WANT_PA), ("stat", sg.WANT_STAT), ("ent", sg.WANT_ENT), ("jnn", sg.WANT_JNN),
                         ("prefix", sg.WANT_PREFIX)):
            tot_ms = 0.0
            for k in range(4):
                ctx.run_device(p0["samples"].data_ptr(), p0["read_off"].data_ptr(), p0["read_len"].data_ptr(),
                               p0["offset"].data_ptr(), p0["unit"].data_ptr(), p0["n_reads"], p0["span"], rna, w_, stream)
                stages = ctx.stage_times()
                ms = sum(m for _, m, _ in stages)
                if k:
                    tot_ms += ms
            ms = tot_ms / 3.0
            by = (6.0 if name == "pa" else 2.0) * p0["n_samples"]  # pa: 2 B in + 4 B out; stat: 2 B in (read 3 times); ent / jnn: 2 B in (jnn reads 3 times)
            siblings[name] = {"ms": ms, "kernels_ms": {n_: round(m_, 4) for n_, m_, _ in stages},
                              "value": p0["n_samples"] / (ms * 1e-3) / 1e9, "unit": UNIT,
                              "algorithmic_gbs": by / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": by / (ms * 1e-3) / 1e9 / measured_peak()[0]}

    # ---- the other BASELINE configs as short sub-lines of the default line (N = 1 only) ---------------------------------
    others = {}
    if world == 1 and args.workload == "dna40k" and not args.no_others:
        del pool[1:]          # (HBM: keep batch 0 for the e2e / svb-zd legs)
        torch.cuda.empty_cache()
        ul = [device_batch(torch, dev, np.full(160, 2_000_000, dtype=np.int64), 0, synth.SEED + 11, 0.1)]
        others["ultralong"] = dict(short_run(torch, sg, local, ul, 0, want),
                                   workload=WORKLOADS["ultralong"].format(mode=args.mode) + " (BASELINE configs[4])")
        st = short_run(torch, sg, local, ul, 0, sg.WANT_STAT)   # `sigtk stat` on the same reads: one CTA per read
        others["ultralong"]["stat"] = {k: st[k] for k in ("value", "unit", "ms_per_step", "stage_ms_per_step")}
        del ul
        torch.cuda.empty_cache()
        rn = [device_batch(torch, dev, lens_all[:8192], 0, synth.SEED + 13, 0.025)]
        others["rna40k"] = dict(short_run(torch, sg, local, rn, 1, want),
                                workload=WORKLOADS["rna40k"].format(mode=args.mode) + " (RNA detector parameters, BASELINE configs[1])")
        del rn
        torch.cuda.empty_cache()
        rb = [real_batch(torch, dev)]
        others["real"] = dict(short_run(torch, sg, local, rb, 0, want), workload=WORKLOADS["real"].format(mode=args.mode),
                              copies=rb[0]["copies"])
        del rb
        torch.cuda.empty_cache()

    # ---- end to end through the host C-ABI: pinned slots, H2D + kernels + D2H per step ----------------------------
    e2e = run_e2e(args, sg, torch, dev, local, pool[0], want, pa_mode, dist, rna, ceiling=True)
    e2e["affinity"] = affinity
    # ---- the same with svb-zd compressed records as input (decoded in HBM), and the decoder alone ------------------
    svb = run_svbzd(args, sg, torch, dev, local, pool[0], want, pa_mode, dist, rna) if not args.no_svbzd else None
    if svb and pa_mode:
        # event-only through the host API: with pA not returned the input side dominates PCIe, which is where the
        # compressed input pays (decoded int16 records vs svb-zd streams, same reads)
        ev_raw = run_e2e(args, sg, torch, dev, local, pool[0], sg.WANT_EVENTS, False, dist, rna, n_reads=max(1, args.e2e_reads // 4))
        ev_svb = run_svbzd(args, sg, torch, dev, local, pool[0], sg.WANT_EVENTS, False, dist, rna)
        svb["event_only"] = {"e2e_int16_records": {k: ev_raw[k] for k in ("value", "h2d_bytes_per_step", "d2h_bytes_per_step")},
                             "e2e_svbzd_streams": {k: ev_svb["e2e"][k] for k in ("value", "h2d_bytes_per_step", "d2h_bytes_per_step")}}

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------------
    peak, peak_src = measured_peak()
    dom = "walk_chunks"
    dom_ms = stage_ms.get(dom, 0.0) / max(args.steps, 1)
    bytes_step = alg_bytes(n_samples, n_reads, n_events, pa_mode) / max(args.steps, 1)
    achieved = bytes_step / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "walk_chunks_bytes_per_sample_pa" if pa_mode else "walk_chunks_bytes_per_sample"  # ncu, profiles/traffic.json
        traffic = float(tj[key]) * n_samples / max(args.steps, 1)
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "walk_chunks_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms_per_launch": dom_ms, "algorithmic_bytes_per_launch": bytes_step,
                "path_frac": bytes_step / (ms_max / max(args.steps, 1) * 1e-3) / 1e9 / peak,
                "stage_ms_per_step": {k: v / max(args.steps, 1) for k, v in stage_ms.items()},
                "stage_timing": "CUDA events on the launch stream, read after every step of an instrumented repeat of the "
                                "K timed steps (same batches, right after the timed region; %.4f ms per step with the "
                                "per-step synchronisation)" % (ms_instrumented / max(args.steps, 1))}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        chk, kind = load_checker()
        n_cpu = min(args.cpu_reads, max(1, int(np.searchsorted(np.cumsum(pool[0]["host_len"]), 80_000_000))))
        reads = host_reads_of(pool[0], n_cpu)
        dt, ns, ne = chk.time_events(reads, rna)
        cpu = {"value": ns / dt / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"first {len(reads)} reads of batch 0 ({ns} samples, {ne} events, {dt:.1f} s)"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload].format(mode=args.mode), "reads_per_step_per_gpu": B_step, "sharding": "contiguous read ranges balanced by samples, no collective",
                       "samples_per_step_per_gpu": n_samples // max(args.steps, 1),
                       "events_per_sample": all_events / max(all_samples, 1.0),
                       "l2": f"inputs {2 * max_span / 1e6:.0f} MB per step > 126 MB L2; pool of {pool_n} distinct batches",
                       "sequential_order_reads": sum(e[1] for e in ev_per_batch),
                       "detector_fixups": sum(e[2] for e in ev_per_batch),
                       "long_detector_replays": sum(e[5] for e in ev_per_batch)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        }
        if svb:
            line["svbzd"] = svb
        if siblings:
            line["siblings"] = siblings
        if others:
            line["other_workloads"] = others
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist:
        dist.destroy_process_group()


DUMP_SEED = 20261020
DUMP_BYTES = 56 << 20


def dump_outputs(ctx, batch, res, pa_mode: bool, out_dir: str) -> None:
    """The result of one device-resident step as .npy files: event counts of every read, and for a seeded sample of
    reads (picked from the read lengths only, so every build picks the same reads) their events and pA. The sample
    takes at most DUMP_BYTES (a read of L samples has at most L // 3 + 1 events of 16 bytes, and 4 bytes of pA a sample).
      read_index   float64[k]    the sampled reads (batch order)
      read_length  float64[k]    their lengths in samples (pa holds them read after read)
      event_count  float64[n]    events of every read of the batch
      event_off    float64[k+1]  the sampled reads' events in event_start / event_mean / event_stdv
      event_start  float64       sample index of each event start
      event_mean   float32, event_stdv float32
      pa           float32       (event+pa mode) the sampled reads' pA samples, read after read"""
    n = batch["n_reads"]
    off, lens = batch["host_off"], batch["host_len"]
    ev_off = ctx.d2h(res.ev_off, np.uint64, n + 1).astype(np.int64)
    picked, budget = [], DUMP_BYTES
    for r in np.random.default_rng(DUMP_SEED).permutation(n)[:256]:
        cost = 4 * int(lens[r]) + 16 * (int(lens[r]) // 3 + 1)
        if cost <= budget:
            picked.append(int(r))
            budget -= cost
    picked = np.sort(np.array(picked, dtype=np.int64))
    a, b = ev_off[picked], ev_off[picked + 1]
    part = lambda ptr, dtype, lo, cnt: ctx.d2h(ptr + np.dtype(dtype).itemsize * int(lo), dtype, int(cnt))
    cat = lambda xs, dtype: np.concatenate(xs) if len(xs) else np.zeros(0, dtype)
    out = {
        "read_index": picked.astype(np.float64),
        "read_length": lens[picked].astype(np.float64),
        "event_count": np.diff(ev_off).astype(np.float64),
        "event_off": np.concatenate([[0], np.cumsum(b - a)]).astype(np.float64),
        "event_start": cat([part(res.ev_start, np.uint32, x, y - x) for x, y in zip(a, b)], np.uint32).astype(np.float64),
        "event_mean": cat([part(res.ev_mean, np.float32, x, y - x) for x, y in zip(a, b)], np.float32),
        "event_stdv": cat([part(res.ev_stdv, np.float32, x, y - x) for x, y in zip(a, b)], np.float32),
    }
    if pa_mode:
        out["pa"] = cat([part(res.pa, np.float32, off[r], lens[r]) for r in picked], np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def run_e2e(args, sg, torch, dev, local, batch, want, pa_mode, dist, rna=0, n_reads=None, ceiling=False):
    """K steps of (pinned slot -> H2D -> kernels -> D2H -> host-visible event table), two slots in flight."""
    B = min(n_reads or args.e2e_reads, batch["n_reads"])
    off, lens = batch["host_off"], batch["host_len"]
    reads = host_reads_of(batch, B)
    span = int(off[B])
    hctx = sg.Context(device=local, max_samples=span + 64, max_reads=B, n_slots=2)
    for s in (0, 1):
        hctx.fill(s, reads, rna)  # the batch loader's job (decode into the pinned slot): outside the timed region
    n_samp = int(lens[:B].sum())

    def wait(slot):
        res = sg._lib.Result()
        hctx._check(hctx._lib.sgpu_wait(hctx._h, slot, C.byref(res)))
        return int(res.n_events)

    hctx.submit(0, want); ne = wait(0)
    hctx.submit(1, want); wait(1)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    steps = max(args.steps, 2)
    t0 = time.perf_counter()
    hctx.submit(0, want)
    for k in range(1, steps):
        hctx.submit(k & 1, want)
        wait((k - 1) & 1)
    wait((steps - 1) & 1)
    dt = time.perf_counter() - t0
    hctx.close()
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(n_samp * steps)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    h2d = 2 * span + 20 * B
    d2h = 12 * ne + 8 * (B + 1) + 8 * B + (4 * span if pa_mode else 0)
    value = float(tot.item()) / float(t.item()) / 1e9
    out = {"value": value, "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "reads_per_step_per_gpu": B, "samples_per_step_per_gpu": n_samp,
           "timing": "host wall clock around submit/wait of K steps, 2 pinned slots in flight, max over ranks; the "
                     "slots are filled once before the timed region (the batch loader's decode into pinned memory is "
                     "not part of this number)"}
    if ceiling:
        # the same bytes, both directions at once, no kernels: what the PCIe links of this box give N ranks
        dt_c = copy_only_ceiling(torch, dev, h2d, d2h, steps, dist)
        cval = float(tot.item()) / dt_c / 1e9
        out["copy_only_ceiling"] = {"value": cval, "unit": UNIT, "frac": value / cval,
                                    "gbs_h2d_plus_d2h": (h2d + d2h) * steps * (int(dist.get_world_size()) if dist else 1) / dt_c / 1e9,
                                    "what": "same h2d/d2h bytes per step from/to pinned memory on two streams, no kernels, max over ranks"}
    return out


def run_svbzd(args, sg, torch, dev, local, batch, want, pa_mode, dist, rna=0):
    """svb-zd compressed records (what a BLOW5 file holds) as the input: (a) end to end through the host C-ABI
    (sgpu_slot_add_read_svbzd: only the compressed bytes cross PCIe), (b) the decoder alone, device resident."""
    B = max(1, min(args.e2e_reads // 4, batch["n_reads"]))
    reads = host_reads_of(batch, B)
    streams = [(synth_mod().svbzd_encode(r[0]), r[1], r[2], r[3]) for r in reads]
    lens = np.array([len(r[0]) for r in reads], dtype=np.int64)
    n_samp = int(lens.sum())
    span = int(((lens + 7) // 8 * 8).sum())
    comp = np.array([len(st[0]) for st in streams], dtype=np.int64)
    hctx = sg.Context(device=local, max_samples=span + 64, max_reads=B, n_slots=2, flags=sg.F_STAGE_TIMERS)
    for s_ in (0, 1):
        hctx.fill_svbzd(s_, streams, rna)

    def wait(slot):
        res = sg._lib.Result()
        hctx._check(hctx._lib.sgpu_wait(hctx._h, slot, C.byref(res)))
        return int(res.n_events)

    hctx.submit(0, want); ne = wait(0)
    hctx.submit(1, want); wait(1)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    steps = max(args.steps, 2)
    t0 = time.perf_counter()
    hctx.submit(0, want)
    for k in range(1, steps):
        hctx.submit(k & 1, want)
        wait((k - 1) & 1)
    wait((steps - 1) & 1)
    dt = time.perf_counter() - t0
    dec_ms = [ms for name, ms, _ in hctx.stage_times() if name == "svbzd_decode"]
    hctx.close()
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(n_samp * steps)], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    comp_bytes = int(((comp + 15) // 16 * 16).sum())
    out = {"e2e": {"value": float(tot.item()) / float(t.item()) / 1e9, "unit": UNIT,
                   "h2d_bytes_per_step": comp_bytes + 32 * B,
                   "d2h_bytes_per_step": 12 * ne + 8 * (B + 1) + 8 * B + (4 * span if pa_mode else 0),
                   "reads_per_step_per_gpu": B, "samples_per_step_per_gpu": n_samp},
           "compressed_bytes_per_sample": float(comp.sum()) / max(n_samp, 1)}
    if dec_ms:  # CUDA events around the decoder's kernels of the last step (stream of the launch)
        ms = dec_ms[0]
        out["decode"] = {"ms": ms, "value": n_samp / (ms * 1e-3) / 1e9, "unit": UNIT,
                         "algorithmic_gbs": (float(comp.sum()) + 2.0 * n_samp) / (ms * 1e-3) / 1e9,
                         "note": "svb_bytes + svb_sums + svb_write + 3 scans; algorithmic bytes = stream in + int16 out"}
    return out


def synth_mod():
    from sigtk_b200 import synth
    return synth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="event+pa", choices=["event+pa", "event"])
    ap.add_argument("--workload", default="dna40k", choices=["dna40k", "dna178k", "ultralong", "rna40k", "real"],
                    help="dna40k = BASELINE.json configs[2] (the headline); the others are reported in DESIGN.md")
    ap.add_argument("--reads-per-step", type=int, default=16384)
    ap.add_argument("--pool", type=int, default=4, help="distinct device-resident batches cycled through")
    ap.add_argument("--e2e-reads", type=int, default=4096)
    ap.add_argument("--cpu-reads", type=int, default=2000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-svbzd", action="store_true", help="skip the compressed-input (svb-zd) measurements")
    ap.add_argument("--no-siblings", action="store_true", help="skip the pa / stat / ent kernel timings")
    ap.add_argument("--no-others", action="store_true", help="skip the ultralong / rna40k / real sub-lines")
    ap.add_argument("--fixed-len", type=int, default=0, help="development: every read of the set has this many samples")
    ap.add_argument("--len-sigma", type=float, default=0.0, help="development: sigma of the lognormal read lengths (default 0.6)")
    ap.add_argument("--chunk-len", type=int, default=0, help="development: samples per detector chunk (0 = automatic)")
    ap.add_argument("--detector-warmup", type=int, default=0, help="development: detector warm-up in samples (0 = default)")
    ap.add_argument("--no-affinity", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

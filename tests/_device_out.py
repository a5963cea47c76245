"""The outputs of a device-resident run (sgpu_run_device and its siblings) copied to the host, read by read where the
layout matters, and their comparison. TEST INFRASTRUCTURE ONLY."""
import numpy as np

import sigtk_b200 as sg


def collect(ctx, d, n, read_off, lens, want, span):
    """the outputs of a device-resident run (device pointers d), per read where the layout matters"""
    out = {}
    if want & sg.WANT_EVENTS:
        out["ev_off"] = ctx.d2h(d.ev_off, np.uint64, n + 1)
        ne = int(out["ev_off"][-1]) if n else 0
        out["ev_start"] = ctx.d2h(d.ev_start, np.uint32, ne)
        out["ev_mean"] = ctx.d2h(d.ev_mean, np.float32, ne).view(np.uint32)
        out["ev_stdv"] = ctx.d2h(d.ev_stdv, np.float32, ne).view(np.uint32)
        out["seq_order"] = ctx.d2h(d.seq_order, np.uint32, n)
        out["fixups"] = ctx.d2h(d.fixups, np.uint32, n)
    if want & sg.WANT_PA:
        flat = ctx.d2h(d.pa, np.float32, span).view(np.uint32)
        out["pa"] = [flat[int(read_off[r]): int(read_off[r]) + int(lens[r])] for r in range(n)]
    if want & sg.WANT_STAT:
        out["stat"] = ctx.d2h(d.stat, np.float32, 6 * n).view(np.uint32)
    if want & sg.WANT_ENT:
        out["ent"] = ctx.d2h(d.ent, np.float64, 3 * n).view(np.uint64)
    if want & sg.WANT_JNN:
        cnt = ctx.d2h(d.jnn_cnt, np.uint32, n)
        seg = ctx.d2h(d.jnn_seg, np.int32, 2 * ((span >> 5) + n + 1)).reshape(-1, 2)
        out["jnn_cnt"] = cnt
        out["jnn"] = [seg[(int(read_off[r]) >> 5) + r: (int(read_off[r]) >> 5) + r + int(cnt[r])] for r in range(n)]
    if want & sg.WANT_PREFIX:
        out["prefix_pos"] = ctx.d2h(d.prefix_pos, np.int32, 4 * n)
        out["prefix_stat"] = ctx.d2h(d.prefix_stat, np.float32, 6 * n).view(np.uint32)
    return out


def assert_same(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, list):
            bad = [r for r in range(len(x)) if not np.array_equal(x[r], y[r])]
            assert not bad, f"{what}: {k} differs for {len(bad)} reads, first {bad[:8]}"
        else:
            assert np.array_equal(x, y), f"{what}: {k} differs"

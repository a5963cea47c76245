"""The caller's own detector parameters (sgpu_set_detector), on the CPU: the oracle's composition orc_pa -> orc_prefix
-> orc_tstat (both windows) -> orc_detect(&set) -> orc_events is getevents for the reference's sets, so it is the truth
for any other set; the streaming reference with the max(w_short, w_long) finality rule reports, over any split, the
whole read's events; and the detector emits its peaks in increasing position order without repeats for every set,
which the event-start bitmap of the batch path rests on."""
import ctypes as C

import numpy as np
import pytest

from _detector_ref import stream_reference, whole_read
from _detector_sets import CUSTOM, REFERENCE
from _live_ref import concat, same_events, split_lengths
from _oracle import Oracle
from _oracle_pa import getevents_pa
from test_live_contract import golden
from sigtk_b200 import synth

SETS = {"dna": REFERENCE[0], "rna": REFERENCE[1], **CUSTOM}
_f32p, _u64p = C.POINTER(C.c_float), C.POINTER(C.c_uint64)


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def reads():
    cb = [synth.make_read_cb(k, n) for k, n in enumerate((1, 5, 13, 27, 28, 29, 600, 7000, 20000))]
    return cb + golden("sp1_dna.npz")[:12] + golden("synth_rna.npz")[:3]


@pytest.mark.parametrize("rna", [0, 1])
def test_composition_is_getevents_for_the_reference_sets(orc, rna):
    rng = np.random.default_rng(3 + rna)
    signals = [orc.pa(*rd) for rd in reads()]
    signals.append((rng.normal(0, 1, 5000) * 1e-3).astype(np.float32))  # sums that round in any order
    for pa in signals:
        assert same_events(whole_read(orc, pa, rna, params=REFERENCE[rna]), getevents_pa(orc, pa, rna)), len(pa)


@pytest.mark.parametrize("name", sorted(SETS))
def test_streaming_is_the_whole_read(orc, name):
    """any split gives the whole read's events; an entry of m samples reports at most the live staging bound of any
    set, ceil((m + 13) / 3) * 2 + 1 events (live_stage_base)"""
    rng = np.random.default_rng(sorted(SETS).index(name))
    for rd in reads():
        pa = orc.pa(*rd)
        whole = whole_read(orc, pa, 0, params=SETS[name])
        if name == "silent":
            assert len(whole[0]) == 1 and int(whole[1][0]) == len(pa)
        for _ in range(2):
            chunks = split_lengths(len(pa), rng)
            got, _ = stream_reference(orc, pa, 0, chunks, params=SETS[name])
            assert same_events(concat(got), whole), (name, len(pa), chunks[:8])
            for m, ev in zip(chunks, got):
                assert len(ev[0]) <= -(-(m + 13) // 3) * 2 + 1


def peaks_of(orc, t1, t2, params):
    s, l = orc.Det(), orc.Det()
    orc.lib.orc_det_init(C.byref(s), C.byref(l))
    p = orc.Params(*params)
    buf = np.empty(len(t1) + 4, np.uint64)
    k = orc.lib.orc_detect(t1.ctypes.data_as(_f32p), t2.ctypes.data_as(_f32p), 0, len(t1), C.byref(p), C.byref(s),
                           C.byref(l), buf.ctypes.data_as(_u64p), buf.shape[0])
    return buf[:k].astype(np.int64)


@pytest.mark.parametrize("name", sorted(SETS))
def test_peaks_come_out_in_increasing_order(orc, name):
    """the emitter reads the peaks from a bitmap: that is the detector's own output only if no peak is emitted before
    an earlier one or twice (the short detector resets the long one while it holds a peak above its threshold,
    events.c:414-422)"""
    params = SETS[name]
    rng = np.random.default_rng(11)
    traces = []
    for _ in range(150):  # t-statistic traces: noise, spikes, plateaus, around both thresholds
        n = 2000
        t = np.abs(rng.normal(0, 1, (2, n))) * rng.choice([0.5, 2.0, 5.0])
        t[:, rng.integers(0, n, 60)] += rng.uniform(0, 12, (2, 60))
        t[:, rng.integers(0, n, 5)] = np.float32(params[2])
        traces.append(t.astype(np.float32))
    for k in range(20):  # step signals through the prefix sums and t-statistics
        lv = np.repeat(rng.uniform(60, 120, 400), rng.integers(2, 30, 400))
        pa = (lv + rng.normal(0, 1 + k % 4, lv.shape[0])).astype(np.float32)
        S, Q = orc.prefix(pa)
        traces.append(np.stack([orc.tstat(S, Q, params[0]), orc.tstat(S, Q, params[1])]).astype(np.float32))
    for t in traces:
        pk = peaks_of(orc, np.ascontiguousarray(t[0]), np.ascontiguousarray(t[1]), params)
        assert np.all(np.diff(pk) > 0), (name, pk[:-1][np.diff(pk) <= 0][:5])

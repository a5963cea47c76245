"""Host-side mirror of the reference's operator interface for the raw-signal path.

The reference works one record at a time through
``float *signal_in_picoamps(slow5_rec_t*)`` (src/sigtk.h:124) and
``event_table getevents(size_t, float*, int8_t rna)`` (src/sigtk.h:134) and
prints ``event_t {start, length, mean, stdv}`` (src/sigtk.h:55-62).  Here the
unit of work is a batch of records; results come back per read in record
order.  All compute happens in ``libsigtk_b200.so`` (hand-written CUDA for
sm_100a) through the C-ABI in ``include/sigtk_b200.h``; this module only moves
numpy buffers in and out of the pinned slots.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (ALIGN, F_DEFAULT, F_FORCE_GENERIC, F_NO_HOST_SLOTS, F_STAGE_TIMERS, LIVE_END, LIVE_RNA, LIVE_START,
                   WANT_EVENTS, WANT_PA, WANT_STAT, WANT_ENT, WANT_JNN, WANT_PREFIX, SgpuError)

Read = Tuple[np.ndarray, float, float, float]  # raw int16, digitisation, offset, range
LiveEntry = Tuple[int, int, np.ndarray, float, float, float]  # channel, LIVE_* flags, raw int16, digitisation, offset,
                                                              # range (the calibration is read with LIVE_START only)
LivePaEntry = Tuple[int, int, np.ndarray]  # channel, LIVE_* flags, pA float32


class Detector(NamedTuple):
    """detector_param (events.c:35-41): the reference's DNA set is Detector(3, 6, 1.4, 9.0, 0.2), its RNA set
    Detector(7, 14, 2.5, 9.0, 1.0)"""
    w_short: int        # window_length1, in [2, 14]
    w_long: int         # window_length2, in [2, 14]
    thr_short: float    # threshold1
    thr_long: float     # threshold2
    peak_height: float


@dataclass
class EventTable:
    """event_table of one read (src/sigtk.h:65-70) as arrays."""
    start: np.ndarray   # uint64
    length: np.ndarray  # float32, (float)(end - start)
    mean: np.ndarray    # float32
    stdv: np.ndarray    # float32

    @property
    def n(self) -> int:
        return int(self.start.shape[0])


@dataclass
class BatchResult:
    n_reads: int
    read_len: np.ndarray
    ev_off: Optional[np.ndarray] = None
    ev_start: Optional[np.ndarray] = None
    ev_mean: Optional[np.ndarray] = None
    ev_stdv: Optional[np.ndarray] = None
    pa: Optional[List[np.ndarray]] = None
    stat: Optional[np.ndarray] = None
    ent: Optional[np.ndarray] = None   # [n_reads][3] float64: raw_ent, delta_ent, byte_ent (ent.c:108-151)
    jnn: Optional[List[np.ndarray]] = None  # per read int64[k][2]: the (x, y) pairs of jnn_raw (jnn.c:269-282)
    prefix_pos: Optional[np.ndarray] = None   # [n_reads][4] int32: adaptor (x, y), poly-A (x, y) (cfunc.c:169-234)
    prefix_stat: Optional[np.ndarray] = None  # [n_reads][6] float32: mean, stdv, median of both stretches' pA
    seq_order: Optional[np.ndarray] = None
    fixups: Optional[np.ndarray] = None

    def events(self, r: int) -> EventTable:
        a, b = int(self.ev_off[r]), int(self.ev_off[r + 1])
        if a == b:  # an empty record has no event
            e = np.empty(0, np.float32)
            return EventTable(np.empty(0, np.uint64), e, e.copy(), e.copy())
        start = self.ev_start[a:b].astype(np.uint64)
        end = np.empty_like(start)
        end[:-1] = start[1:]
        end[-1] = self.read_len[r]
        length = (end - start).astype(np.float32)
        return EventTable(start, length, self.ev_mean[a:b].copy(), self.ev_stdv[a:b].copy())


def live_tables(ev_off, ev_start, ev_len, ev_mean, ev_stdv) -> List[EventTable]:
    """one EventTable per entry of a live run (start: sample index in the channel's read)"""
    out = []
    for e in range(len(ev_off) - 1):
        a, b = int(ev_off[e]), int(ev_off[e + 1])
        out.append(EventTable(ev_start[a:b].astype(np.uint64), ev_len[a:b].astype(np.float32), ev_mean[a:b].copy(),
                              ev_stdv[a:b].copy()))
    return out


def _np_from(ptr: int, dtype, count: int) -> np.ndarray:
    if count == 0:
        return np.empty(0, dtype=dtype)
    buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=count).copy()


class Context:
    """One GPU context (sgpu_ctx_t)."""

    def __init__(self, device: int = 0, max_samples: int = 1 << 24, max_reads: int = 1 << 16,
                 n_slots: int = 2, flags: int = F_DEFAULT):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.max_samples, self.max_reads, self.n_slots = max_samples, max_reads, n_slots
        rc = self._lib.sgpu_create(C.byref(self._h), device, max_samples, max_reads, n_slots, flags)
        if rc != 0:
            raise SgpuError(rc, self._lib.sgpu_strerror(rc).decode())

    def close(self) -> None:
        if self._h:
            self._lib.sgpu_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc < 0:
            raise SgpuError(rc, f"{self._lib.sgpu_strerror(rc).decode()} | {self._lib.sgpu_last_error(self._h).decode()}")

    # ---- host path -------------------------------------------------------
    def fill(self, slot: int, reads: Sequence[Read], rna: int) -> None:
        self._check(self._lib.sgpu_slot_reset(self._h, slot, int(rna)))
        for raw, dig, off, rng in reads:
            raw = np.ascontiguousarray(raw, dtype=np.int16)
            rc = self._lib.sgpu_slot_add_read(self._h, slot, raw.ctypes.data, raw.shape[0], float(dig), float(off),
                                              float(rng))
            self._check(int(rc))

    def fill_svbzd(self, slot: int, reads: Sequence, rna: int) -> None:
        """reads: (svb-zd stream uint8[], digitisation, offset, range) -- the record's raw_signal field as slow5lib
        stores it with SLOW5_COMPRESS_SVB_ZD; the samples are decoded in HBM"""
        self._check(self._lib.sgpu_slot_reset(self._h, slot, int(rna)))
        for st, dig, off, rng in reads:
            st = np.ascontiguousarray(st, dtype=np.uint8)
            rc = self._lib.sgpu_slot_add_read_svbzd(self._h, slot, st.ctypes.data, st.shape[0], float(dig), float(off),
                                                    float(rng))
            self._check(int(rc))

    def fill_pa(self, slot: int, signals: Sequence[np.ndarray], rna: int) -> None:
        """signals: float32 pA arrays, one per record (getevents(n, pa, rna) on the caller's own signal); a slot holds
        max_samples / 2 of them"""
        self._check(self._lib.sgpu_slot_reset(self._h, slot, int(rna)))
        for pa in signals:
            pa = np.ascontiguousarray(pa, dtype=np.float32)
            self._check(int(self._lib.sgpu_slot_add_read_pa(self._h, slot, pa.ctypes.data, pa.shape[0])))

    def run_pa(self, signals: Sequence[np.ndarray], rna: int = 0, want: int = WANT_EVENTS, slot: int = 0) -> BatchResult:
        """fill_pa + submit + wait: the event tables of records given as pA floats"""
        self.fill_pa(slot, signals, rna)
        self.submit(slot, want)
        return self.wait(slot, want)

    def run_svbzd(self, reads: Sequence, rna: int = 0, want: int = WANT_EVENTS, slot: int = 0) -> BatchResult:
        self.fill_svbzd(slot, reads, rna)
        self.submit(slot, want)
        return self.wait(slot, want)

    def decode_svbzd_device(self, bytes_ptr: int, n_bytes: int, comp_off_ptr: int, comp_len_ptr: int, read_off_ptr: int,
                            read_len_ptr: int, n_reads: int, n_blocks: int, samples_out_ptr: int, stream: int = 0) -> None:
        sb = _lib.SvbDevBatch(bytes_ptr, n_bytes, comp_off_ptr, comp_len_ptr, read_off_ptr, read_len_ptr, n_reads,
                              n_blocks)
        self._check(self._lib.sgpu_decode_svbzd_device(self._h, C.byref(sb), C.c_void_p(samples_out_ptr),
                                                       C.c_void_p(stream)))

    def submit(self, slot: int, want: int) -> None:
        self._check(self._lib.sgpu_submit(self._h, slot, want))

    def wait(self, slot: int, want: int) -> BatchResult:
        res = _lib.Result()
        self._check(self._lib.sgpu_wait(self._h, slot, C.byref(res)))
        pb = C.POINTER(_lib.Batch)()
        self._check(self._lib.sgpu_slot_batch(self._h, slot, C.byref(pb)))
        b = pb.contents
        n = int(b.n_reads)
        read_len = np.ctypeslib.as_array(b.read_len, shape=(max(n, 1),))[:n].copy()
        read_off = np.ctypeslib.as_array(b.read_off, shape=(n + 1,)).copy()
        out = BatchResult(n_reads=n, read_len=read_len)
        if want & WANT_EVENTS:
            ne = int(res.n_events)
            out.ev_off = _np_from(res.ev_off, np.uint64, n + 1)
            out.ev_start = _np_from(res.ev_start, np.uint32, ne)
            out.ev_mean = _np_from(res.ev_mean, np.float32, ne)
            out.ev_stdv = _np_from(res.ev_stdv, np.float32, ne)
            out.seq_order = _np_from(res.seq_order, np.uint32, n)
            out.fixups = _np_from(res.fixups, np.uint32, n)
        if want & WANT_STAT:
            out.stat = _np_from(res.stat, np.float32, n * 6).reshape(n, 6)
        if want & WANT_ENT:
            out.ent = _np_from(res.ent, np.float64, n * 3).reshape(n, 3)
        if want & WANT_JNN:
            cnt = _np_from(res.jnn_cnt, np.uint32, n)
            span = int(read_off[n]) if n else 0
            seg = _np_from(res.jnn_seg, np.int32, 2 * ((span >> 5) + n + 1)).reshape(-1, 2)
            out.jnn = []
            for r in range(n):
                base = (int(read_off[r]) >> 5) + r  # SGPU_JNN_BASE
                out.jnn.append(seg[base: base + int(cnt[r])].astype(np.int64))
        if want & WANT_PREFIX:
            out.prefix_pos = _np_from(res.prefix_pos, np.int32, n * 4).reshape(n, 4)
            out.prefix_stat = _np_from(res.prefix_stat, np.float32, n * 6).reshape(n, 6)
        if want & WANT_PA:
            span = int(read_off[n]) if n else 0
            flat = _np_from(res.pa, np.float32, span)
            out.pa = [flat[int(read_off[r]): int(read_off[r]) + int(read_len[r])].copy() for r in range(n)]
        return out

    def run(self, reads: Sequence[Read], rna: int = 0, want: int = WANT_EVENTS, slot: int = 0) -> BatchResult:
        """fill + submit + wait on one slot (the call a host program makes per batch)."""
        self.fill(slot, reads, rna)
        self.submit(slot, want)
        return self.wait(slot, want)

    # ---- live event detection: signal in chunks, detector state per channel in HBM -----------------------------
    def live_open(self, n_channels: int) -> None:
        """sgpu_live_open: the table of n_channels channels (once per context)"""
        self._check(self._lib.sgpu_live_open(self._h, int(n_channels)))

    def live_fill(self, slot: int, entries: Sequence[LiveEntry]) -> None:
        self._check(self._lib.sgpu_slot_reset(self._h, slot, 0))
        for ch, flags, raw, dig, off, rng in entries:
            raw = np.ascontiguousarray(raw, dtype=np.int16)
            self._check(int(self._lib.sgpu_slot_add_live(self._h, slot, int(ch), int(flags), raw.ctypes.data,
                                                         raw.shape[0], float(dig), float(off), float(rng))))

    def live_fill_pa(self, slot: int, entries: Sequence[LivePaEntry]) -> None:
        """live entries given as pA floats (sgpu_slot_add_live_pa); a slot holds max_samples / 2 of them"""
        self._check(self._lib.sgpu_slot_reset(self._h, slot, 0))
        for ch, flags, pa in entries:
            pa = np.ascontiguousarray(pa, dtype=np.float32)
            self._check(int(self._lib.sgpu_slot_add_live_pa(self._h, slot, int(ch), int(flags), pa.ctypes.data,
                                                            pa.shape[0])))

    def live_wait(self, slot: int) -> List[EventTable]:
        """the events of a submitted live slot of either form, entry by entry"""
        res = _lib.LiveResult()
        self._check(self._lib.sgpu_wait_live(self._h, slot, C.byref(res)))
        pb = C.POINTER(_lib.Batch)()
        self._check(self._lib.sgpu_slot_batch(self._h, slot, C.byref(pb)))
        n, ne = int(pb.contents.n_reads), int(res.n_events)
        return live_tables(_np_from(res.ev_off, np.uint64, n + 1), _np_from(res.ev_start, np.uint32, ne),
                           _np_from(res.ev_len, np.uint32, ne), _np_from(res.ev_mean, np.float32, ne),
                           _np_from(res.ev_stdv, np.float32, ne))

    def live_push(self, entries: Sequence[LiveEntry], slot: int = 0) -> List[EventTable]:
        """one push of live entries (at most one per channel): fill + submit + wait; -> the events each entry reports"""
        self.live_fill(slot, entries)
        self.submit(slot, WANT_EVENTS)
        return self.live_wait(slot)

    def live_push_pa(self, entries: Sequence[LivePaEntry], slot: int = 0) -> List[EventTable]:
        """one push of live entries of pA floats (at most one per channel); -> the events each entry reports"""
        self.live_fill_pa(slot, entries)
        self.submit(slot, WANT_EVENTS)
        return self.live_wait(slot)

    def run_device_live(self, samples_ptr: int, read_off_ptr: int, read_len_ptr: int, channel_ptr: int, flags_ptr: int,
                        offset_ptr: int, unit_ptr: int, n_entries: int, span: int, stream: int = 0) -> _lib.LiveResult:
        """sgpu_run_device_live: live entries already in device memory; -> device pointers of the events (the count
        is counters()["n_events"] once the stream is done)"""
        db = _lib.DevLiveBatch(samples_ptr, read_off_ptr, read_len_ptr, channel_ptr, flags_ptr, offset_ptr, unit_ptr,
                               n_entries, span)
        res = _lib.LiveResult()
        self._check(self._lib.sgpu_run_device_live(self._h, C.byref(db), C.c_void_p(stream), C.byref(res)))
        return res

    def run_device_live_pa(self, pa_ptr: int, read_off_ptr: int, read_len_ptr: int, channel_ptr: int, flags_ptr: int,
                           n_entries: int, span: int, stream: int = 0) -> _lib.LiveResult:
        """sgpu_run_device_live_pa: live entries of pA floats already in device memory; -> device pointers of the
        events, as run_device_live"""
        db = _lib.DevLivePaBatch(pa_ptr, read_off_ptr, read_len_ptr, channel_ptr, flags_ptr, n_entries, span)
        res = _lib.LiveResult()
        self._check(self._lib.sgpu_run_device_live_pa(self._h, C.byref(db), C.c_void_p(stream), C.byref(res)))
        return res

    # ---- device-resident path ---------------------------------------------
    def run_device(self, samples_ptr: int, read_off_ptr: int, read_len_ptr: int, offset_ptr: int, unit_ptr: int,
                   n_reads: int, span: int, rna: int, want: int, stream: int = 0) -> _lib.Result:
        db = _lib.DevBatch(samples_ptr, read_off_ptr, read_len_ptr, offset_ptr, unit_ptr, n_reads, int(rna), span)
        res = _lib.Result()
        self._check(self._lib.sgpu_run_device(self._h, C.byref(db), want, C.c_void_p(stream), C.byref(res)))
        return res

    def run_device_pa(self, pa_ptr: int, read_off_ptr: int, read_len_ptr: int, n_reads: int, span: int, rna: int,
                      want: int = WANT_EVENTS, stream: int = 0) -> _lib.Result:
        """sgpu_run_device_pa: events of pA floats already in device memory (read_off multiples of ALIGN)"""
        db = _lib.DevPaBatch(pa_ptr, read_off_ptr, read_len_ptr, n_reads, int(rna), span)
        res = _lib.Result()
        self._check(self._lib.sgpu_run_device_pa(self._h, C.byref(db), want, C.c_void_p(stream), C.byref(res)))
        return res

    def d2h(self, dev_ptr: int, dtype, count: int) -> np.ndarray:
        """copy `count` items of a device result array (a pointer from run_device) to a new numpy array"""
        out = np.empty(count, dtype=dtype)
        self._check(self._lib.sgpu_memcpy_d2h(self._h, out.ctypes.data, C.c_void_p(dev_ptr), out.nbytes))
        return out

    def stage_times(self) -> list:
        """[(name, ms, launches)] of the last run (context created with F_STAGE_TIMERS)"""
        arr = (_lib.StageTime * 16)()
        n = self._lib.sgpu_stage_times(self._h, arr, 16)
        self._check(n)
        return [(arr[k].name.decode(), float(arr[k].ms), int(arr[k].launches)) for k in range(n)]

    def counters(self) -> dict:
        c = _lib.Counters()
        self._check(self._lib.sgpu_counters(self._h, C.byref(c)))
        return {"n_events": int(c.n_events), "n_seq_order_reads": int(c.n_seq_order_reads),
                "n_fixups": int(c.n_fixups), "n_kernel_launches": int(c.n_kernel_launches), "status": int(c.status),
                "n_long_jobs": int(c.n_long_jobs)}

    def set_detector(self, det: Optional[Detector]) -> None:
        """sgpu_set_detector: every later event detection of the context (batches, device-resident runs, live reads
        started from now on) uses `det`; None restores the reference's sets, chosen by rna"""
        if det is None:
            self._check(self._lib.sgpu_set_detector(self._h, None))
            return
        p = _lib.DetectorParams(int(det[0]), int(det[1]), float(det[2]), float(det[3]), float(det[4]))
        self._check(self._lib.sgpu_set_detector(self._h, C.byref(p)))

    def set_param(self, key: int, value: float) -> None:
        """development / test parameters (_lib.PARAM_*): chunk length, detector warm-up, the long detector's threshold"""
        self._check(self._lib.sgpu_set_param(self._h, int(key), float(value)))


# ---- per-record conveniences mirroring the reference's function names --------
def signal_in_picoamps(ctx: Context, raw: np.ndarray, digitisation: float, offset: float, range_: float) -> np.ndarray:
    """misc.c:15-32 for one record."""
    return ctx.run([(raw, digitisation, offset, range_)], 0, WANT_PA).pa[0]


def getevents(ctx: Context, raw: np.ndarray, digitisation: float, offset: float, range_: float,
              rna: int = 0) -> EventTable:
    """events.c:553-573 for one record (pA conversion is fused, so this takes the raw samples)."""
    return ctx.run([(raw, digitisation, offset, range_)], rna, WANT_EVENTS).events(0)


def getevents_pa(ctx: Context, pa: np.ndarray, rna: int = 0) -> EventTable:
    """events.c:553-573 for one record given as pA floats, exactly as the reference's getevents(n, pa, rna)."""
    return ctx.run_pa([pa], rna, WANT_EVENTS).events(0)


def stat(ctx: Context, raw: np.ndarray, digitisation: float, offset: float, range_: float) -> np.ndarray:
    """The six numbers of stat_func (cfunc.c:126-159) for one record."""
    return ctx.run([(raw, digitisation, offset, range_)], 0, WANT_STAT).stat[0]


def ent(ctx: Context, raw: np.ndarray) -> np.ndarray:
    """raw_ent, delta_ent, byte_ent of one record as `sigtk ent` prints them (ent.c:108-151)."""
    return ctx.run([(raw, 8192.0, 0.0, 1.0)], 0, WANT_ENT).ent[0]


def jnn_raw(ctx: Context, raw: np.ndarray, rna: int = 0) -> np.ndarray:
    """jnn_raw (jnn.c:269-282) with jnn_print's parameters for one record: int64[k][2] (x, y) pairs."""
    return ctx.run([(raw, 8192.0, 0.0, 1.0)], rna, WANT_JNN).jnn[0]

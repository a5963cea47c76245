"""The slot rules of the host path, kind by kind: a slot holds one kind of record (int16 records, svb-zd streams, pA
records or live entries) from sgpu_slot_reset to sgpu_wait / sgpu_wait_live, each kind computes its own set of
products, and each append refuses a record that can never fit (SGPU_E_TOOBIG) before one that does not fit now
(SGPU_E_FULL)."""
import ctypes as C

import numpy as np
import pytest

from _oracle import Oracle
import sigtk_b200 as sg
from sigtk_b200 import _lib

pytestmark = pytest.mark.gpu

E_INVAL, E_FULL, E_TOOBIG, E_STATE = -1, -4, -5, -6
START, END = sg.LIVE_START, sg.LIVE_END
MAX_SAMPLES, MAX_READS, N_CHANNELS = 4096, 8, 8
KINDS = ("int16", "svbzd", "pa", "live")
ALL_WANTS = set(range(1, 64))
ALLOWED = {"none": ALL_WANTS, "int16": ALL_WANTS, "svbzd": ALL_WANTS, "pa": {sg.WANT_EVENTS},
           "live": {sg.WANT_EVENTS}}

RAW = np.random.default_rng(3).normal(500, 60, 100).astype(np.int16)
PA = np.linspace(60.0, 90.0, 100).astype(np.float32)


@pytest.fixture(scope="module")
def ctx():
    with sg.Context(device=0, max_samples=MAX_SAMPLES, max_reads=MAX_READS) as c:
        c.live_open(N_CHANNELS)
        yield c


@pytest.fixture(scope="module")
def stream():
    return Oracle().svbzd_encode(RAW)


def add(ctx, stream, kind, slot=0, channel=0):
    """appends one small record of `kind` to the slot; -> the return code"""
    lib, h = ctx._lib, ctx._h
    if kind == "int16":
        return lib.sgpu_slot_add_read(h, slot, RAW.ctypes.data, RAW.size, 8192.0, 4.0, 1400.0)
    if kind == "svbzd":
        return lib.sgpu_slot_add_read_svbzd(h, slot, stream.ctypes.data, stream.size, 8192.0, 4.0, 1400.0)
    if kind == "pa":
        return lib.sgpu_slot_add_read_pa(h, slot, PA.ctypes.data, PA.size)
    # a whole read per entry, so that every push leaves the channel closed
    return lib.sgpu_slot_add_live(h, slot, channel, START | END, RAW.ctypes.data, RAW.size, 8192.0, 4.0, 1400.0)


def fill(ctx, stream, kind, slot=0):
    assert ctx._lib.sgpu_slot_reset(ctx._h, slot, 0) == 0
    if kind != "none":
        assert add(ctx, stream, kind, slot) == 0


def wait(ctx, kind, slot=0):
    if kind == "live":
        return ctx._lib.sgpu_wait_live(ctx._h, slot, C.byref(_lib.LiveResult()))
    return ctx._lib.sgpu_wait(ctx._h, slot, C.byref(_lib.Result()))


@pytest.mark.parametrize("first", KINDS)
def test_one_kind_per_slot(ctx, stream, first):
    for second in KINDS:
        fill(ctx, stream, first)
        want = 1 if second == first else E_STATE
        assert add(ctx, stream, second, channel=1) == want, (first, second)
        assert ctx._lib.sgpu_slot_reset(ctx._h, 0, 0) == 0
        assert add(ctx, stream, second) == 0, (first, second)   # a reset slot takes every kind
    assert ctx._lib.sgpu_slot_reset(ctx._h, 0, 0) == 0


@pytest.mark.parametrize("kind", KINDS)
def test_submitted_slot_refuses_everything(ctx, stream, kind):
    lib, h = ctx._lib, ctx._h
    fill(ctx, stream, kind)
    assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == 0
    for other in KINDS:
        assert add(ctx, stream, other, channel=2) == E_STATE, other
    assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == E_STATE
    assert lib.sgpu_slot_reset(h, 0, 0) == E_STATE
    assert wait(ctx, kind) == 0
    assert wait(ctx, kind) == E_STATE
    assert lib.sgpu_slot_reset(h, 0, 0) == 0


@pytest.mark.parametrize("kind", ("none",) + KINDS)
def test_wants_of_each_kind(ctx, stream, kind):
    lib, h = ctx._lib, ctx._h
    for want in range(64):
        fill(ctx, stream, kind)
        rc = lib.sgpu_submit(h, 0, want)
        if want in ALLOWED[kind]:
            assert rc == 0, (kind, want)
            assert wait(ctx, kind) == 0, (kind, want)
        else:
            assert rc == E_INVAL, (kind, want)
            assert wait(ctx, kind) == E_STATE, (kind, want)


def test_wait_matches_the_kind(ctx, stream):
    lib, h = ctx._lib, ctx._h
    for kind in ("none",) + KINDS:
        fill(ctx, stream, kind)
        assert lib.sgpu_wait(h, 0, C.byref(_lib.Result())) == E_STATE, kind            # not submitted
        assert lib.sgpu_wait_live(h, 0, C.byref(_lib.LiveResult())) == E_STATE, kind
        assert lib.sgpu_submit(h, 0, sg.WANT_EVENTS) == 0
        if kind == "live":
            assert lib.sgpu_wait(h, 0, C.byref(_lib.Result())) == E_STATE
        else:
            assert lib.sgpu_wait_live(h, 0, C.byref(_lib.LiveResult())) == E_STATE, kind
        assert wait(ctx, kind) == 0, kind                                            # (still submitted)
        assert wait(ctx, kind) == E_STATE, kind


def fake_stream(n, n_bytes):
    """a stream header for n samples, n_bytes long (the appends check only the header against the length)"""
    s = np.zeros(max(n_bytes, 4), np.uint8)
    s[:4] = np.array([n], np.uint32).view(np.uint8)
    return s


def test_capacity_boundaries(ctx):
    lib, h = ctx._lib, ctx._h
    big = np.zeros(MAX_SAMPLES + 64, np.int16)
    bigf = np.zeros(MAX_SAMPLES, np.float32)

    def reset():
        assert lib.sgpu_slot_reset(h, 0, 0) == 0

    def raw(n):
        return lib.sgpu_slot_add_read(h, 0, big.ctypes.data, n, 8192.0, 4.0, 1400.0)

    def pa(n):
        return lib.sgpu_slot_add_read_pa(h, 0, bigf.ctypes.data, n)

    def live(n, channel=0, flags=START):
        return lib.sgpu_slot_add_live(h, 0, channel, flags, big.ctypes.data, n, 8192.0, 4.0, 1400.0)

    def svb(s, n_bytes=None):
        return lib.sgpu_slot_add_read_svbzd(h, 0, s.ctypes.data, s.size if n_bytes is None else n_bytes, 8192.0, 4.0,
                                            1400.0)

    # int16 records and live entries: max_samples, every record padded to 8; 2^31 samples never
    for add1 in (raw, lambda n: live(n, 0)):
        reset()
        assert add1(MAX_SAMPLES + 1) == E_TOOBIG
        assert add1(1 << 31) == E_TOOBIG
        assert add1(MAX_SAMPLES - 7) == 0         # max_samples with its padding
        assert add1(1) == E_FULL                  # (live: before the second entry of channel 0)
        assert add1(MAX_SAMPLES + 1) == E_TOOBIG
    reset()
    for r in range(MAX_READS):
        assert raw(0) == r
    assert raw(0) == E_FULL
    reset()
    for r in range(MAX_READS):
        assert live(0, r % N_CHANNELS) == r
    assert live(0, 0) == E_FULL
    # live: the channel and the flags before the length, the second entry of a channel after it
    reset()
    assert live(1 << 31, N_CHANNELS) == E_INVAL
    assert live(1 << 31, 0, START | 8) == E_INVAL
    assert live(MAX_SAMPLES - 8, 0) == 0
    assert live(16, 0) == E_FULL
    assert live(MAX_SAMPLES + 1, 0) == E_TOOBIG
    assert live(0, 0) == E_INVAL
    assert live(0, 1) == 1
    # pA records: max_samples / 2 floats, 2^32 never
    reset()
    assert pa(MAX_SAMPLES // 2 + 1) == E_TOOBIG
    assert pa(1 << 32) == E_TOOBIG
    assert pa((1 << 31) + 8) == E_TOOBIG
    assert pa(MAX_SAMPLES // 2 - 7) == 0
    assert pa(1) == E_FULL
    assert pa(MAX_SAMPLES // 2 + 1) == E_TOOBIG
    reset()
    for r in range(MAX_READS):
        assert pa(0) == r
    assert pa(0) == E_FULL
    # svb-zd streams: the samples as int16 records, and comp_cap = 2 * max_samples bytes of streams (16-byte padding)
    comp_cap = 2 * MAX_SAMPLES
    n_max = 4 + (1000 + 3) // 4 + 4 * 1000          # the longest stream 1000 samples can have
    reset()
    assert svb(fake_stream(MAX_SAMPLES + 1, 4 + (MAX_SAMPLES + 4) // 4 + MAX_SAMPLES + 1)) == E_TOOBIG
    assert svb(fake_stream(3000, comp_cap + 1)) == E_TOOBIG
    assert svb(fake_stream(1 << 30, 0), 1 << 32) == E_TOOBIG                        # over 2^32 - 1 bytes
    assert svb(fake_stream(1000, 10)) == -9                                           # shorter than its header says
    assert svb(fake_stream(1000, n_max + 1)) == -9
    assert svb(fake_stream(1000, n_max)) == 0                                         # 4,256 bytes with its padding
    assert svb(fake_stream(1000, comp_cap - 4256 + 1)) == E_FULL                      # the bytes do not fit
    assert svb(fake_stream(1000, comp_cap - 4256)) == 1
    assert svb(fake_stream(1000, 4 + 250 + 1000)) == E_FULL                           # the samples fit, the bytes not
    reset()
    assert svb(fake_stream(MAX_SAMPLES, 4 + MAX_SAMPLES // 4 + MAX_SAMPLES)) == 0
    assert svb(fake_stream(1, 4 + 1 + 1)) == E_FULL                                   # the samples do not fit
    # a stream over comp_cap in a slot that is full of samples: TOOBIG, not FULL
    assert svb(fake_stream(3000, comp_cap + 1)) == E_TOOBIG
    assert svb(fake_stream(1 << 30, 0), 1 << 32) == E_TOOBIG
    reset()

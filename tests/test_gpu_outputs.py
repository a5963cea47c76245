"""The per-batch outputs of the C-ABI as a whole (include/sigtk_b200.h, sgpu_result_t), called through ctypes so that
the library's own rules are tested, not those of the Python mirror:
- sgpu_wait returns exactly the arrays of the wanted products, and every product's arrays do not depend on which
  other products the batch asked for, on which slot it ran or on what ran in the other slot meanwhile;
- a batch of empty records, and one without reads, give every output its defined value;
- sgpu_run_device always returns the arrays allocated with the context and the others only when wanted."""
import ctypes as C

import numpy as np
import pytest

from sigtk_b200 import _lib, synth

pytestmark = pytest.mark.gpu

EVENTS, PA, STAT, ENT, JNN, PREFIX = (_lib.WANT_EVENTS, _lib.WANT_PA, _lib.WANT_STAT, _lib.WANT_ENT, _lib.WANT_JNN,
                                      _lib.WANT_PREFIX)
PRODUCTS = (EVENTS, PA, STAT, ENT, JNN, PREFIX)
ALL = 63
# the result fields of every product
FIELDS = {EVENTS: ("ev_off", "ev_start", "ev_mean", "ev_stdv", "seq_order", "fixups"), PA: ("pa",), STAT: ("stat",),
          ENT: ("ent",), JNN: ("jnn_cnt", "jnn_seg"), PREFIX: ("prefix_pos", "prefix_stat")}
EAGER = FIELDS[EVENTS] + FIELDS[STAT]  # allocated with the context


def batch(seed):
    """Seeded DNA reads: an empty record, reads shorter than the 2,000-sample window of `prefix` and longer ones."""
    rng = np.random.default_rng(seed)
    lens = [int(n) for n in rng.integers(2001, 40000, 6)] + [0, 1500, 7, 1999]
    rng.shuffle(lens)
    return [synth.make_read(i, n, seed) if n else (np.zeros(0, np.int16), synth.DIGITISATION, 0.0, synth.RANGE)
            for i, n in enumerate(lens)]


class Ctx:
    def __init__(self, flags=0, n_slots=2):
        self.lib = _lib.load()
        self.h = C.c_void_p()
        assert self.lib.sgpu_create(C.byref(self.h), 0, 1 << 20, 64, n_slots, flags) == 0

    def close(self):
        self.lib.sgpu_destroy(self.h)

    def fill(self, slot, reads):
        assert self.lib.sgpu_slot_reset(self.h, slot, 0) == 0
        for raw, dig, off, rng in reads:
            raw = np.ascontiguousarray(raw, dtype=np.int16)
            assert self.lib.sgpu_slot_add_read(self.h, slot, raw.ctypes.data, raw.shape[0], dig, off, rng) >= 0

    def submit(self, slot, want):
        assert self.lib.sgpu_submit(self.h, slot, want) == 0

    def wait(self, slot):
        res = _lib.Result()
        assert self.lib.sgpu_wait(self.h, slot, C.byref(res)) == 0
        pb = C.POINTER(_lib.Batch)()
        assert self.lib.sgpu_slot_batch(self.h, slot, C.byref(pb)) == 0
        n = int(pb.contents.n_reads)
        off = np.ctypeslib.as_array(pb.contents.read_off, shape=(n + 1,)).copy()
        lens = np.ctypeslib.as_array(pb.contents.read_len, shape=(max(n, 1),))[:n].copy()
        return res, outputs(res, off, lens, int(res.n_events), host_array)

    def run(self, reads, want, slot=0):
        self.fill(slot, reads)
        self.submit(slot, want)
        return self.wait(slot)

    def d2h(self, ptr, dtype, count):
        out = np.empty(count, dtype=dtype)
        assert self.lib.sgpu_memcpy_d2h(self.h, out.ctypes.data, C.c_void_p(ptr), out.nbytes) == 0
        return out


def host_array(ptr, dtype, count):
    if count == 0:
        return np.empty(0, dtype)
    return np.frombuffer((C.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr), dtype, count).copy()


def outputs(res, off, lens, n_events, fetch):
    """{field: bytes} of every non-NULL field, restricted to what the batch defines (the samples of every read for pa,
    the segments of every read for jnn_seg)"""
    n = len(lens)
    got = {}
    for name, dtype, count in (("ev_off", np.uint64, n + 1), ("ev_start", np.uint32, n_events),
                               ("ev_mean", np.float32, n_events), ("ev_stdv", np.float32, n_events),
                               ("seq_order", np.uint32, n), ("fixups", np.uint32, n), ("stat", np.float32, 6 * n),
                               ("ent", np.float64, 3 * n), ("jnn_cnt", np.uint32, n),
                               ("prefix_pos", np.int32, 4 * n), ("prefix_stat", np.float32, 6 * n)):
        if getattr(res, name):
            got[name] = fetch(getattr(res, name), dtype, count).tobytes()
    span = int(off[n])
    if res.pa:
        pa = fetch(res.pa, np.float32, span)
        got["pa"] = b"".join(pa[off[r]:off[r] + lens[r]].tobytes() for r in range(n))
    if res.jnn_seg:
        seg = fetch(res.jnn_seg, np.int32, 2 * ((span >> 5) + n + 1)).reshape(-1, 2)
        cnt = np.frombuffer(got["jnn_cnt"], np.uint32)
        got["jnn_seg"] = b"".join(seg[(int(off[r]) >> 5) + r:][:int(cnt[r])].tobytes() for r in range(n))
    return got


def non_null(res):
    return {name for names in FIELDS.values() for name in names if getattr(res, name)}


def wanted_fields(want):
    return {name for p in PRODUCTS if want & p for name in FIELDS[p]}


@pytest.fixture(scope="module")
def ctx():
    c = Ctx()
    yield c
    c.close()


def test_every_want_mask_returns_its_products_unchanged(ctx):
    reads = batch(11)
    single = {}
    for p in PRODUCTS:
        res, got = ctx.run(reads, p)
        assert non_null(res) == wanted_fields(p)
        single.update(got)
    assert single["ev_off"] != bytes(len(single["ev_off"])) and single["jnn_seg"]
    pos = np.frombuffer(single["prefix_pos"], np.int32).reshape(-1, 4)
    assert (pos[:, 1] == -1).any() and (pos[:, 1] != -1).any()  # records within the window and longer ones
    for want in range(1, ALL + 1):
        res, got = ctx.run(reads, want)
        assert non_null(res) == wanted_fields(want), f"want {want}"
        assert res.n_events == (len(np.frombuffer(single["ev_start"], np.uint32)) if want & EVENTS else 0)
        for name, val in got.items():
            assert val == single[name], f"want {want}: {name} differs from the run that wants only its product"


def test_two_slots_in_flight_with_different_masks():
    reads = [batch(21), batch(22)]
    c = Ctx()
    try:
        got = {}
        for masks in ((JNN, PREFIX | PA), (PREFIX | PA, JNN)):
            for slot in (0, 1):
                c.fill(slot, reads[slot])
                c.submit(slot, masks[slot])
            for slot in (0, 1):
                res, out = c.wait(slot)
                assert non_null(res) == wanted_fields(masks[slot])
                got[slot, masks[slot]] = out
        for slot in (0, 1):
            single = {}
            for p in (JNN, PREFIX, PA):
                single.update(c.run(reads[slot], p)[1])
            for mask in (JNN, PREFIX | PA):
                for name, val in got[slot, mask].items():
                    assert val == single[name], f"slot {slot}, want {mask}: {name}"
    finally:
        c.close()


def test_empty_batches_give_the_defined_values(ctx):
    ctx.run(batch(31), ALL)
    empty = (np.zeros(0, np.int16), synth.DIGITISATION, 0.0, synth.RANGE)
    res, got = ctx.run([empty] * 3, ALL)
    assert res.n_events == 0 and non_null(res) == wanted_fields(ALL)
    expect = {"ev_off": np.zeros(4, np.uint64), "seq_order": np.zeros(3, np.uint32), "fixups": np.zeros(3, np.uint32),
              "stat": np.zeros(18, np.float32), "ent": np.zeros(9, np.float64), "jnn_cnt": np.zeros(3, np.uint32),
              "prefix_pos": np.full(12, -1, np.int32), "prefix_stat": np.zeros(18, np.float32)}
    for name, val in expect.items():
        assert got[name] == val.tobytes(), name
    assert got["pa"] == b"" and got["jnn_seg"] == b""
    res, got = ctx.run([], ALL)
    assert res.n_events == 0 and got["ev_off"] == np.zeros(1, np.uint64).tobytes()


def test_device_path_returns_eager_outputs_always_and_lazy_ones_when_wanted(ctx):
    torch = pytest.importorskip("torch")
    reads = batch(41)
    lens = np.array([len(r[0]) for r in reads], dtype=np.int64)
    off = np.zeros(len(reads) + 1, dtype=np.int64)
    off[1:] = np.cumsum((lens + 7) // 8 * 8)
    flat = np.zeros(int(off[-1]), dtype=np.int16)
    for r, rd in enumerate(reads):
        flat[off[r]:off[r] + lens[r]] = rd[0]
    dev = torch.device("cuda:0")
    d_s = torch.from_numpy(flat).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    d_o = torch.tensor([np.float32(r[2]) for r in reads], dtype=torch.float32, device=dev)
    d_u = torch.tensor([np.float32(r[3]) / np.float32(r[1]) for r in reads], dtype=torch.float32, device=dev)
    db = _lib.DevBatch(d_s.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_o.data_ptr(), d_u.data_ptr(), len(reads),
                       0, int(off[-1]))
    dctx = Ctx(flags=_lib.F_NO_HOST_SLOTS, n_slots=0)
    try:
        for p in PRODUCTS:
            res = _lib.Result()
            assert dctx.lib.sgpu_run_device(dctx.h, C.byref(db), p, None, C.byref(res)) == 0
            torch.cuda.synchronize()
            assert non_null(res) == set(EAGER) | wanted_fields(p), f"want {p}"
            assert res.n_events == 0
            c = _lib.Counters()
            assert dctx.lib.sgpu_counters(dctx.h, C.byref(c)) == 0 and c.status == 0
            got = outputs(res, off, lens, int(c.n_events), dctx.d2h)
            host = ctx.run(reads, p)[1]
            for name in wanted_fields(p):
                assert got[name] == host[name], f"want {p}: {name} differs from the host path"
    finally:
        dctx.close()

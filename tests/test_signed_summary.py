"""The signed float-order summaries of float_order.cuh (tile_summary_signed, sgn_then, sgn_fits) restated in numpy
float32 and checked against the sequential loop s <- fl(s + v) on random signed tiles: wherever a composition of tile
summaries is accepted, the accumulator it gives is the sequential one bit for bit. Runs on the CPU."""
import numpy as np

F = np.float32
P = 12582912                                    # 1.5 * 2^23
FAR = 1 << 28


def scale_of(s):
    e = int(np.frexp(np.float64(s))[1]) - 1
    return F(np.copysign(2.0 ** (23 - e), s))


def tile_summary(row, scale):
    """-> (inc, lo, hi) per parity of the incoming mantissa, or None when the tile cannot be summarised"""
    out = []
    with np.errstate(all="ignore"):
        x = (np.asarray(row, F) * scale).astype(F)
        for p in (0, 1):
            path = np.add.accumulate(np.concatenate([[F(P + p)], x]).astype(F), dtype=F)[1:]
            if not (np.all(path > F(2.0 ** 23)) and np.all(path < F(2.0 ** 24))):
                return None
            out.append((int(path[-1]) - P - p, int(path.min()) - P - p, int(path.max()) - P - p))
    return out


def then(a, b):
    c = []
    for p in (0, 1):
        d = a[p][0]
        q = (p ^ d) & 1
        c.append((d + b[q][0], min(a[p][1], d + b[q][1]), max(a[p][2], d + b[q][2])))
    return c


def fits(u, S):
    p = S & 1
    return S + u[p][1] >= 0x800001 and S + u[p][2] <= 0xFFFFFF


def mantissa(s):
    m, e = np.frexp(np.float64(abs(s)))
    return int(m * 2 ** 24), e


def test_composed_summaries_are_the_sequential_sum():
    rng = np.random.default_rng(2718)
    accepted = 0
    for case in range(600):
        n_tiles = int(rng.integers(1, 33))
        mag = 10.0 ** rng.uniform(-3, 4)
        x = rng.normal(rng.uniform(-0.5, 0.5) * mag, mag, 32 * n_tiles).astype(F)
        if case % 5 == 0:
            x = (np.round(x * 8) / 8).astype(F)  # half and quarter ulps of the accumulator: ties of both parities
        if case % 7 == 0:
            x[rng.integers(0, len(x), 5)] = F(-0.0)
        s = F(rng.choice([-1, 1]) * 10.0 ** rng.uniform(0, 6) * mag)
        seq = np.add.accumulate(np.concatenate([[s], x]).astype(F), dtype=F)[32::32]   # after every tile
        scale = scale_of(s)
        S, e = mantissa(s)
        u = [(0, FAR, -FAR)] * 2
        for t in range(n_tiles):
            v = tile_summary(x[32 * t:32 * t + 32], scale)
            if v is None:
                break
            u = then(u, v)
            if not fits(u, S):
                break
            S_after = S + u[S & 1][0]
            got = F(np.copysign(np.ldexp(np.float64(S_after), e - 24), s))
            assert got.view(np.uint32) == seq[t].view(np.uint32), (case, t)
            accepted += 1
    assert accepted > 3000

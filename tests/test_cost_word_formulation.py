"""The 16-bit cost word of the materialised path, restated in numpy (no GPU).

When every worker's ext_ask_price is <= 0xFFFE the build kernel writes one 16-bit word per (ask, worker) pair instead of
the int64 key price << 32 | worker:
    word = price + b * (0xFFFF - price),  b = 1 when the pair is infeasible (the predicate's sign bit)
and a lane forms the two 32-bit halves of its 4-column store with one multiply-add per worker:
    half = b1 * ((0xFFFF - p1) << 16) + (b0 * (0xFFFF - p0) + (p0 | p1 << 16)).
The argmin folds each row on the 32-bit key price << 16 | column offset within the CTA's span (offsets lane-relative
while folding, the lane's base added once per row) and widens it to the int64 key only at the per-CTA flush.  These
tests check that the word, widened, is the oracle's int64 cost and that the 32-bit fold picks the int64 minimum.
"""
import numpy as np
import pytest

from oracle import pm_oracle as orc
from protocol_b200 import synth

INF = np.int64(0x7FFFFFFFFFFFFFFF)
M32 = np.uint64(0xFFFFFFFF)


def words_from_fail(b, price):
    """b: (T, W) 0/1 infeasible; price: (W,) <= 0xFFFE -> (T, W) uint16 words."""
    b = b.astype(np.uint32)
    p = price.astype(np.uint32)[None, :]
    return (b * (np.uint32(0xFFFF) - p) + p).astype(np.uint16)


def packed_halves(b, price):
    """The kernel's pair form: one 32-bit half per two adjacent columns (W even), computed modulo 2^32."""
    b = b.astype(np.uint64)
    p = price.astype(np.uint64)
    b0, b1, p0, p1 = b[:, 0::2], b[:, 1::2], p[None, 0::2], p[None, 1::2]
    d0 = np.uint64(0xFFFF) - p0
    d1s = ((np.uint64(0xFFFF) - p1) << np.uint64(16)) & M32
    return ((b1 * d1s + ((b0 * d0 + (p0 | (p1 << np.uint64(16)))) & M32)) & M32).astype(np.uint32)


def widen(words, w0=0):
    """pm_widen_cost: price << 32 | worker, or INF for the infeasible word."""
    h = words.astype(np.int64)
    cols = np.arange(words.shape[1], dtype=np.int64) + w0
    return np.where(words == 0xFFFF, INF, (h << 32) | cols[None, :])


def priced_tables(price, n_asks=240, n_workers=2050, shift=0):
    w = synth.make_workers(n_workers, seed=synth.SEED_WORKERS + 40 + shift, price=price)
    a = synth.make_asks(n_asks, "mixed", seed=synth.SEED_ASKS + 40 + shift)
    bits, npat, nmod, words = synth.intern_tables(w, a)
    return w, a, bits, words


@pytest.mark.parametrize("price", ["loguniform", "zipf"])
def test_widened_words_equal_the_oracle_cost(price):
    w, a, bits, words = priced_tables(price)
    T, W = len(a), len(w)
    cost = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, 0, T, 0, W, threads=8, want_cost=True)["cost"]
    pr = w.b["ext_ask_price"].astype(np.uint32)
    assert pr.max() <= 0xFFFE and len(np.unique(pr)) > 50
    fail = cost == INF
    assert 0 < fail.mean() < 1
    words16 = words_from_fail(fail, pr)
    assert np.array_equal(widen(words16), cost)
    # the packed pair form writes the same bytes as the per-column form (little-endian: even column in the low half)
    halves = packed_halves(fail, pr)
    assert np.array_equal(halves.view(np.uint16).reshape(T, W), words16)


def test_widened_words_of_a_shard_carry_the_global_worker_index():
    w, a, bits, words = priced_tables("loguniform", n_asks=60, n_workers=3000, shift=1)
    w0, w1 = 1100, 2900
    cost = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, 0, len(a), w0, w1, threads=8, want_cost=True)["cost"]
    words16 = words_from_fail(cost == INF, w.b["ext_ask_price"][w0:w1])
    assert np.array_equal(widen(words16, w0), cost)


def test_boundary_prices():
    p = np.array([0, 1, 0x7FFF, 0x8000, 0xFFFD, 0xFFFE], dtype=np.uint32)
    for b in (0, 1):
        bb = np.full((1, len(p)), b)
        got = words_from_fail(bb, p)[0]
        assert np.array_equal(got, np.full(len(p), 0xFFFF) if b else p)
        assert np.array_equal(packed_halves(bb, p).view(np.uint16)[0], got)


def test_key_order_equals_int64_order():
    """price << 16 | offset orders exactly like price << 32 | (base + offset) for price <= 0xFFFE, offset < 65536."""
    rng = np.random.default_rng(7)
    n = 2_000_000
    edges = np.array([0, 1, 0x7FFF, 0x8000, 0xFFFD, 0xFFFE], dtype=np.uint64)
    p = np.concatenate([rng.integers(0, 0xFFFF, n, dtype=np.uint64), np.repeat(edges, 4)])
    o = np.concatenate([rng.integers(0, 65536, n, dtype=np.uint64), np.tile(np.array([0, 1, 65534, 65535], np.uint64), 6)])
    k32 = (p << np.uint64(16)) | o
    assert k32.max() < 0xFFFF0000   # below every infeasible key
    for base in (0, 1 << 20, 0xFFFFFFFF - 65535):
        k64 = ((p << np.uint64(32)) | (np.uint64(base) + o)).astype(np.int64)
        assert (k64 >= 0).all()
        i, j = rng.integers(0, len(p), (2, n))
        assert np.array_equal(np.sign(k32[i].astype(np.int64) - k32[j].astype(np.int64)),
                              np.sign(k64[i] - k64[j]))
        assert np.array_equal(np.argsort(k32, kind="stable"), np.argsort(k64, kind="stable"))


def fold_like_the_kernel(words, S=4, warps=8):
    """pm_argmin16's fold of one row of a CTA's span: per lane S loads of 8 words, lane-relative key offsets, the lane's
    base added once, then the minimum over lanes and warps.  -> (min 32-bit key, feasible count)."""
    span = warps * S * 256
    assert words.shape == (span,)
    best_all, cnt = 0xFFFFFFFF, 0
    for warp in range(warps):
        for lane in range(32):
            lane_off = warp * S * 256 + lane * 8
            best = 0xFFFF0000
            for s in range(S):
                x8 = words[lane_off + s * 256: lane_off + s * 256 + 8].astype(np.uint32)
                for j in range(4):
                    x = int(x8[2 * j]) | (int(x8[2 * j + 1]) << 16)
                    off = s * 256 + 2 * j
                    klo = (x * 65536 + off) & 0xFFFFFFFF
                    khi = (x & 0xFFFF0000) | (off + 1)
                    best = min(best, klo, khi)
                    cnt += (klo < 0xFFFF0000) + (x < 0xFFFF0000)
            best += lane_off
            assert best <= 0xFFFFFFFF
            best_all = min(best_all, best)
    return best_all, cnt


@pytest.mark.parametrize("frac_feasible", [0.0, 0.0005, 0.3, 1.0])
def test_argmin_fold_picks_the_int64_minimum(frac_feasible):
    rng = np.random.default_rng(int(frac_feasible * 1e4) + 3)
    span, cta_c0, w0 = 8 * 4 * 256, 3 * 8192, 5000
    # few price levels: many ties in price, so the column order decides
    price = rng.choice(np.array([7, 9, 0xFFFE, 12], np.uint16), span)
    feas = rng.random(span) < frac_feasible
    words = np.where(feas, price, np.uint16(0xFFFF)).astype(np.uint16)
    key, cnt = fold_like_the_kernel(words)
    assert cnt == int(feas.sum())
    wide = widen(words[None, :], w0 + cta_c0)[0]
    if cnt:
        got = ((key >> 16) << 32) | (w0 + cta_c0 + (key & 0xFFFF))
        assert got == int(wide.min())
    else:
        assert key >= 0xFFFF0000

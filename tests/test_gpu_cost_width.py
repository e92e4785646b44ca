"""The materialised pass with a 16-bit cost tile against the int64 one (PM_TUNE_COST=8) and the oracle.

The engine writes 16-bit price words (2 B per evaluation) when the fast predicate applies and every worker's
ext_ask_price is <= 0xFFFE, else int64 keys (8 B); stats.cost_bytes_written tells which one ran.  Every fetch() array
must be identical between the two widths, and equal to the oracle's."""
import os

import numpy as np
import pytest

from helpers import groups_equal
from oracle import pm_oracle as orc
from protocol_b200 import abi, synth
from protocol_b200.engine import Engine

pytestmark = pytest.mark.gpu

MAT = abi.PM_MODE_FIRST_FIT | abi.PM_PATH_MATERIALIZED
FIELDS = ("worker_group", "worker_ask", "group_ask", "group_off", "group_members", "ask_best", "ask_count")


def make_engine(wide: bool, tile_bytes: int):
    if wide:
        os.environ["PM_TUNE_COST"] = "8"   # read at pm_create
    try:
        return Engine(cost_tile_bytes=tile_bytes)
    finally:
        os.environ.pop("PM_TUNE_COST", None)


def tables(n_asks, n_workers, price, shift=0, kind="mixed"):
    w = synth.make_workers(n_workers, seed=synth.SEED_WORKERS + 60 + shift, price=price)
    a = synth.make_asks(n_asks, kind, seed=synth.SEED_ASKS + 60 + shift, group_sizes=[(1, 1), (2, 2), (1, 3)])
    bits, npat, nmod, words = synth.intern_tables(w, a)
    return w, a, bits, npat, nmod, words


def load(eng, w, a, bits, npat, nmod, words):
    eng.set_asks(a.asks, a.opts)
    eng.set_model_table(bits, npat, nmod, words)
    eng.set_workers(w.a, w.b)


def run(t, wide, tile_bytes=1 << 20, shard=None):
    eng = make_engine(wide, tile_bytes)
    load(eng, *t)
    if shard is not None:
        eng.set_shard(*shard)
    eng.match(MAT)
    res = eng.fetch()
    eng.close()
    return res


def bytes_per_eval(res):
    st = res.stats
    assert st["cost_bytes_read"] == st["cost_bytes_written"]
    return st["cost_bytes_written"] / st["evals"]


def check_against_oracle(res, t, w0=0, nw=None):
    w, a, bits, _, _, words = t
    nw = len(w) - w0 if nw is None else nw
    ev = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, 0, len(a), w0, w0 + nw, threads=8)
    assert np.array_equal(res.ask_best, ev["row_best"])
    assert np.array_equal(res.ask_count, ev["row_count"])


def same_outputs(r16, r64):
    for f in FIELDS:
        assert np.array_equal(getattr(r16, f), getattr(r64, f)), f


@pytest.mark.parametrize("price,n_asks,n_workers,tile_bytes", [
    ("loguniform", 700, 9000, 1 << 20),       # several tiles: 1 MiB holds 128 rows of 9216 int64 keys
    ("zipf", 700, 9000, 64 << 20),
    ("loguniform", 1, 5000, 1 << 20),         # nt = 1
    ("zipf", 300, 700, 64 << 10),             # nw < 1024, tiles of 8 rows
    ("loguniform", 1500, 3333, 256 << 10),    # nw not a multiple of 1024, tiles of 64 rows
])
def test_16bit_tile_equals_int64_tile_and_oracle(price, n_asks, n_workers, tile_bytes):
    t = tables(n_asks, n_workers, price, shift=n_workers % 97)
    r16, r64 = run(t, False, tile_bytes), run(t, True, tile_bytes)
    assert bytes_per_eval(r16) == 2 and bytes_per_eval(r64) == 8
    same_outputs(r16, r64)
    check_against_oracle(r16, t)
    w, a, bits, _, _, words = t
    og = orc.soa_form_groups(w.a, w.b, a.asks, a.opts, bits, words)
    assert groups_equal(r16, og)
    if tile_bytes < 64 << 20:
        assert r16.stats["n_tiles"] > 1 or n_asks == 1


def test_shard_with_nonzero_first_worker():
    t = tables(500, 7000, "zipf", shift=5)
    shard = (2500, 3100)
    r16, r64 = run(t, False, 1 << 20, shard), run(t, True, 1 << 20, shard)
    assert bytes_per_eval(r16) == 2 and bytes_per_eval(r64) == 8
    same_outputs(r16, r64)
    check_against_oracle(r16, t, *shard)


@pytest.mark.parametrize("top,expect", [(0xFFFE, 2), (0xFFFF, 8), (0x10000, 8)])
def test_price_boundary(top, expect):
    """0xFFFE is the largest price a 16-bit word holds (0xFFFF means infeasible); beyond it the int64 tile runs."""
    w, a, bits, npat, nmod, words = tables(400, 4000, "loguniform", shift=9)
    b = w.b.copy()
    b["ext_ask_price"][::7] = top                      # many workers at the boundary, some of them feasible
    b["ext_ask_price"][1::11] = top - 1
    w.b = b
    t = (w, a, bits, npat, nmod, words)
    res = run(t, False)
    assert bytes_per_eval(res) == expect
    check_against_oracle(res, t)
    og = orc.soa_form_groups(w.a, w.b, a.asks, a.opts, bits, words)
    assert groups_equal(res, og)


def test_prices_from_2_pow_31_run_the_int64_tile():
    """Prices >= 2^31 take the int64 tile, the same one PM_TUNE_COST=8 runs.  (Their keys are negative as int64; the
    int64 argmin merges row minima as unsigned in shared memory, so its ask_best there is not the oracle's signed
    minimum — a property of the int64 kernel, not of the tile width.)"""
    w, a, bits, npat, nmod, words = tables(400, 4000, "loguniform", shift=9)
    b = w.b.copy()
    b["ext_ask_price"][::7] = 0x80000000
    w.b = b
    t = (w, a, bits, npat, nmod, words)
    r, r64 = run(t, False), run(t, True)
    assert bytes_per_eval(r) == 8
    same_outputs(r, r64)


def test_price_change_between_passes_switches_width():
    w, a, bits, npat, nmod, words = tables(600, 6000, "loguniform", shift=13)
    t = (w, a, bits, npat, nmod, words)
    eng = make_engine(False, 1 << 20)
    load(eng, *t)
    eng.match(MAT)
    first = eng.fetch()
    assert bytes_per_eval(first) == 2
    check_against_oracle(first, t)
    for price, expect in ((0x10000, 8), (5, 2)):
        k = 4321
        b = w.b.copy()
        b["ext_ask_price"][k] = price
        w.b = b
        eng.upsert_workers(w.a[k:k + 1].copy(), b[k:k + 1].copy(), first=k)
        eng.match(MAT)
        res = eng.fetch()
        assert bytes_per_eval(res) == expect
        check_against_oracle(res, (w, a, bits, npat, nmod, words))
    eng.close()


@pytest.mark.parametrize("price", ["loguniform", "zipf"])
def test_cost_tile_on_priced_tables(price):
    """pm_build_cost_tile runs the 16-bit build and widens it: the int64 rows equal the oracle's cost matrix."""
    w, a, bits, npat, nmod, words = tables(300, 5000, price, shift=17)
    for wide in (False, True):
        eng = make_engine(wide, 1 << 20)
        load(eng, w, a, bits, npat, nmod, words)
        cost = eng.cost_tile(100, 150)
        eng.close()
        ref = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, 100, 250, 0, len(w), threads=8, want_cost=True)["cost"]
        assert np.array_equal(cost, ref)

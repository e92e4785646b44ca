"""The worker-sharded pass (SURVEY 8e) on hardware, through the C ABI.

* One GPU: several engines, each on its own contiguous share of the worker table (pm_set_shard), run
  pm_match_local; the three exchange buffers are merged the way the collective merges them (concatenate / min / sum)
  and every engine runs pm_match_finish.  Groups must equal the unsharded engine's and the CPU oracle's.
* Two or more GPUs in one process (pm_multi: NCCL all-gather inside the library): same check.  Skipped on a
  machine with one GPU.
"""
import numpy as np
import pytest

from helpers import groups_equal, load_engine
from oracle import pm_oracle as orc
from protocol_b200 import abi, synth
from protocol_b200.engine import Engine, MultiEngine
from protocol_b200.sharded import shard_range, wrap_device_buffers

pytestmark = pytest.mark.gpu

SIZES = [(1, 1), (2, 2), (2, 4), (3, 3), (4, 8), (1, 3), (5, 16)]


def tables(n_asks, n_workers, group_sizes=None, seed_shift=0, kind="mixed", price=None):
    w = synth.make_workers(n_workers, seed=synth.SEED_WORKERS + seed_shift, with_addresses=n_workers <= 20000, price=price)
    a = synth.make_asks(n_asks, kind, seed=synth.SEED_ASKS + seed_shift, group_sizes=group_sizes)
    bits, npat, nmod, words = synth.intern_tables(w, a)
    return w, a, dict(asks=a.asks, opts=a.opts, wa=w.a, wb=w.b, bits=bits, n_patterns=npat, n_models=nmod, words=words,
                      lat=w.lat, lon=w.lon)


def sharded_pass_on_one_gpu(t, n_shards, mode, addr_rank=None, locations=False):
    """n_shards engines on device 0; the exchange done here, as the collective does it."""
    import torch

    W, T = len(t["wa"]), len(t["asks"])
    engs, bufs, ranges = [], [], []
    for r in range(n_shards):
        lo, hi = shard_range(W, n_shards, r)
        e = Engine(cost_tile_bytes=1 << 20)
        load_engine(e, t, addr_rank=addr_rank, locations=locations)
        e.set_shard(lo, hi - lo)
        e.match_local(mode)
        e.sync()
        engs.append(e)
        bufs.append(wrap_device_buffers(e, W, T))
        ranges.append((lo, hi))
    first = torch.cat([bufs[r][0][lo:hi] for r, (lo, hi) in enumerate(ranges)])
    best = torch.stack([b[1] for b in bufs]).min(dim=0).values
    cnt = torch.stack([b[2] for b in bufs]).sum(dim=0).to(torch.int32)
    # outside its own range a shard's first_ask must still be "none": nothing was evaluated there
    for r, (lo, hi) in enumerate(ranges):
        fa = bufs[r][0]
        assert bool((fa[:lo] == -1).all()) and bool((fa[hi:] == -1).all())
    results = []
    for r, e in enumerate(engs):
        bufs[r][0].copy_(first)
        bufs[r][1].copy_(best)
        bufs[r][2].copy_(cnt)
        torch.cuda.synchronize()
        e.match_finish(mode)
        results.append(e.fetch())
    for e in engs:
        e.close()
    return results


@pytest.mark.parametrize("n_shards", [2, 3])
@pytest.mark.parametrize("path", [abi.PM_PATH_MATERIALIZED, abi.PM_PATH_FUSED], ids=["materialized", "fused"])
def test_sharded_first_fit_equals_unsharded_and_oracle(n_shards, path):
    """First-fit with group sizes > 1 (the tail sweep runs on the merged arrays) and a ragged last shard."""
    w, a, t = tables(300, 10007, group_sizes=SIZES, seed_shift=11)
    mode = abi.PM_MODE_FIRST_FIT | path
    og = orc.soa_form_groups(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"], addr_rank=w.addr_rank)
    ev = orc.soa_eval_matrix(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"], 0, 300, 0, 10007, threads=8)
    whole = Engine()
    load_engine(whole, t, addr_rank=w.addr_rank)
    whole.match(mode)
    ref = whole.fetch()
    whole.close()
    assert groups_equal(ref, og)
    for res in sharded_pass_on_one_gpu(t, n_shards, mode, addr_rank=w.addr_rank):
        assert groups_equal(res, og), "sharded groups differ from the oracle"
        assert np.array_equal(res.worker_group, ref.worker_group) and np.array_equal(res.worker_ask, ref.worker_ask)
        assert np.array_equal(res.ask_best, ev["row_best"]) and np.array_equal(res.ask_count, ev["row_count"])
        assert res.stats["n_bumped"] == ref.stats["n_bumped"] > 0


@pytest.mark.parametrize("n_shards", [2, 3])
def test_sharded_proximity_solo_equals_oracle(n_shards):
    """Proximity policy with solo groups: located workers first inside every configuration (mod.rs:526-530)."""
    w, a, t = tables(200, 9001, seed_shift=5)
    mode = abi.PM_MODE_PROXIMITY
    og = orc.soa_form_groups(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"], lat=t["lat"], lon=t["lon"],
                             proximity=True)
    for res in sharded_pass_on_one_gpu(t, n_shards, mode, locations=True):
        assert groups_equal(res, og)


def test_shard_wider_than_table_and_empty_shards():
    """More shards than workers: trailing shards are empty and contribute nothing."""
    w, a, t = tables(17, 5, seed_shift=3)
    og = orc.soa_form_groups(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"])
    for res in sharded_pass_on_one_gpu(t, 7, abi.PM_MODE_FIRST_FIT):
        assert groups_equal(res, og)


def _n_devices():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("mode,sizes", [(abi.PM_MODE_FIRST_FIT, SIZES), (abi.PM_MODE_FIRST_FIT | abi.PM_PATH_FUSED, SIZES),
                                        (abi.PM_MODE_PROXIMITY, None)], ids=["first_fit", "first_fit_fused", "proximity_solo"])
def test_multi_engine_in_one_process(mode, sizes):
    """pm_multi on every visible GPU: NCCL all-gather inside the library, result on device 0 == oracle."""
    n = _n_devices()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    w, a, t = tables(500, 40003, group_sizes=sizes, seed_shift=23)
    prox = (mode & 0xFF) == abi.PM_MODE_PROXIMITY
    og = orc.soa_form_groups(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"], addr_rank=None,
                             lat=t["lat"], lon=t["lon"], proximity=prox)
    ev = orc.soa_eval_matrix(t["wa"], t["wb"], t["asks"], t["opts"], t["bits"], t["words"], 0, 500, 0, 40003, threads=8)
    m = MultiEngine(list(range(n)), cost_tile_bytes=4 << 20, timing=True)
    m.set_asks(t["asks"], t["opts"])
    m.set_model_table(t["bits"], t["n_patterns"], t["n_models"], t["words"])
    m.set_workers(t["wa"], t["wb"])
    if prox:
        m.set_locations(t["lat"], t["lon"])
    for _ in range(3):   # repeated passes reuse the communicators and buffers
        m.match(mode)
        res = m.fetch()
        assert groups_equal(res, og)
        assert np.array_equal(res.ask_best, ev["row_best"]) and np.array_equal(res.ask_count, ev["row_count"])
    st = [m.stats(i) for i in range(n)]
    assert sum(s["evals"] for s in st) == 500 * 40003          # the evaluation was split, not replicated
    assert all(s["exchange_bytes"] > 0 for s in st)
    m.close()

"""The one-sweep slot sort and the hot-run kernels at their boundaries: engine vs CPU oracle, bit-exact.

Sort pipeline (GCRA_FLAG_SORT_PATH): batch sizes around the sort tile (4096 keys), full-size ticks, slot-bit counts
that give one, two and three sort passes, and hot keys whose run lengths sit on the thresholds of the hot-run
kernels (LONG_RUN_MIN = 256: one CTA per run, GIANT_RUN_MIN = 4096: one cluster per run).  Index-order pipeline
(GCRA_FLAG_INDEX_PATH): batches whose sorted residue is empty, one row, and exactly one sort tile."""
import numpy as np
import pytest

import oracle
import throttlecrab_b200 as tc
import traces
from throttlecrab_b200._native import FLAG_INDEX_PATH, FLAG_SORT_PATH, FLAG_TIGHT_TABLE
from gpu_util import engine_requests, first_mismatch

# the flags choose the pipeline, so the suite-wide run over the three GCRA_INDEX_MIN settings is not needed
pytestmark = [pytest.mark.gpu, pytest.mark.parametrize("k1_path", ["auto"], indirect=True)]

SORT_TILE = 4096
LONG_RUN_MIN, GIANT_RUN_MIN = 256, 4096


def _replay(req, capacity, batch, flags, max_batch=None):
    st_o = oracle.OracleStore(oracle.PERIODIC, capacity=capacity, created_ns=traces.T0, p0=10**9)
    want = st_o.replay(req)
    st_e = tc.ManualStore(capacity=capacity, created_ns=traces.T0, max_batch=max_batch or batch, flags=flags)
    lim = tc.RateLimiter(st_e)
    ereq = engine_requests(req)
    got = np.empty(len(req), tc.RES_DTYPE)
    for a in range(0, len(req), batch):
        lim.rate_limit_batch(ereq[a:a + batch], out=got[a:a + batch])
    assert first_mismatch(want, got, req) is None, first_mismatch(want, got, req)
    assert st_e.len() == st_o.len()
    return st_e


def _rows(keys, rng, t_step=(0, 0, 1000, 20_000_000)):
    """Requests on `keys` in the given order: mixed policies and quantities, a slowly advancing clock."""
    n = len(keys)
    req = np.zeros(n, traces.REQ_DTYPE)
    req["key"] = keys
    traces.fill_policy(req, (req["key"] % np.uint64(8)).astype(np.int64))
    req["quantity"] = rng.choice([0, 1, 1, 1, 2, 5], n)
    req["now_ns"] = traces.T0 + np.cumsum(rng.choice(t_step, n))
    return req


@pytest.mark.parametrize("batch", [256, SORT_TILE - 1, SORT_TILE, SORT_TILE + 1, 3 * SORT_TILE + 7])
def test_sort_pipeline_batch_sizes_around_the_tile(batch):
    n_keys = 5000
    req = np.concatenate([traces.warm_pass(n_keys), traces.config2(n_keys=n_keys, n_ticks=4, tick_size=batch)])
    _replay(req, capacity=n_keys, batch=batch, flags=FLAG_SORT_PATH)


@pytest.mark.parametrize("tick", [1 << 20, 1 << 21])
def test_sort_pipeline_full_size_ticks(tick):
    n_keys = 200_000
    req = np.concatenate([traces.warm_pass(n_keys), traces.config2(n_keys=n_keys, n_ticks=2, tick_size=tick)])
    st = _replay(req, capacity=n_keys, batch=tick, flags=FLAG_SORT_PATH)
    assert st.stats()["index_batches"] == 0


@pytest.mark.parametrize("capacity", [16, 20_000])
def test_sort_pipeline_tight_table_pass_counts(capacity):
    """GCRA_FLAG_TIGHT_TABLE: 64 slots growing (one pass of 6+ bits), 2^15 slots (two passes)."""
    rng = np.random.default_rng(11)
    n = 60_000
    keys = (rng.integers(0, 20_000, n) * np.linspace(0.05, 1.0, n)).astype(np.uint64)
    req = _rows(keys, rng)
    st = _replay(req, capacity=capacity, batch=4096, flags=FLAG_SORT_PATH | FLAG_TIGHT_TABLE)
    if capacity == 16:
        assert st.stats()["grows"] >= 1


def test_sort_pipeline_one_giant_run():
    """Every request of the batch on one key: one sorted run, decided by the cluster kernel."""
    rng = np.random.default_rng(12)
    req = _rows(np.full(3 * GIANT_RUN_MIN + 5, 7, np.uint64), rng)
    _replay(req, capacity=100, batch=len(req), flags=FLAG_SORT_PATH)


def test_sort_pipeline_run_lengths_on_the_hot_run_thresholds():
    rng = np.random.default_rng(13)
    runs = {1: LONG_RUN_MIN - 1, 2: LONG_RUN_MIN, 3: GIANT_RUN_MIN - 1, 4: GIANT_RUN_MIN}
    keys = np.concatenate([np.full(c, k, np.uint64) for k, c in runs.items()] +
                          [np.arange(100, 3100, dtype=np.uint64)])
    keys = keys[rng.permutation(len(keys))]
    req = _rows(keys, rng)
    _replay(req, capacity=4000, batch=len(req), flags=FLAG_SORT_PATH)


@pytest.mark.parametrize("residue", [0, 1, SORT_TILE])
def test_index_pipeline_residue_sizes(residue):
    """Fresh keys, quantity 1: every key's first request creates its entry (a state change), so exactly the
    repeats of a key go to the sorted residue."""
    rng = np.random.default_rng(14)
    n = 8192
    keys = np.arange(n, dtype=np.uint64)
    keys[n - residue:] = keys[:residue]            # `residue` keys occur twice
    keys = keys[rng.permutation(n)]
    req = np.zeros(n, traces.REQ_DTYPE)
    req["key"] = keys
    traces.fill_policy(req, np.zeros(n, np.int64))
    req["quantity"] = 1
    req["now_ns"] = traces.T0
    st = _replay(req, capacity=n, batch=n, flags=FLAG_INDEX_PATH)
    assert st.stats()["index_batches"] == 1

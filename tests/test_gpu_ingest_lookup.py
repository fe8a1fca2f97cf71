"""The two-pass ingest's tile loads and table lookups at their edges, forced on for every launch (FLAG_TWO_PASS_ALWAYS):

  pass 2: a key set crafted so that twelve keys of one dictionary bucket share one home group of the aggregation
          table (four slots: the group overflows into the following slots) and five of them also share the 5-bit tag
          (several candidates per lookup, told apart by the key confirm)
  pass 1: device batches whose columns are sliced at an odd row (not 16-byte aligned: those tiles load row by row
          instead of by TMA) beside aligned ones in the same launch, and batches whose last tile is partial.

Host batches are checked against the oracle; device batches against an independent group-by (torch.unique +
index_add, which wraps like i64 SUM)."""
import ctypes as C

import numpy as np
import pytest

from oracle import arroyo_oracle as O
from tests.test_gpu_parity import S, SUM_AVG, T0, assert_same, gen_stream, run_both

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    from tests import gpu_ops
    return gpu_ops


def _p2_group_tag(keys):
    """The aggregation table's home group and tag of each key (ingest_two_pass.cuh: p2_hash / p2_group / p2_tag)."""
    h = (keys.astype(np.uint64) * np.uint64(0xD6E8FEB86659FD93)) >> np.uint64(32)
    tag = (h >> np.uint64(4)) & np.uint64(31)
    return h >> np.uint64(21), np.where(tag == 0, np.uint64(1), tag)


def _bucket(keys, n_buckets):
    """The dictionary bucket of each key (bdict.cuh: bd_hash / bd_bucket)."""
    k = keys.astype(np.uint64)
    h = (k ^ (k >> np.uint64(32))) * np.uint64(0x9E3779B97F4A7C15)
    return ((h >> np.uint64(32)) * np.uint64(n_buckets)) >> np.uint64(32)


def colliding_keys(n_buckets, n_group=12, n_tag=5):
    """`n_group` keys of bucket 0 with one home group, `n_tag` of them with one tag too."""
    cand = np.arange(1, 1 << 22, dtype=np.int64)
    with np.errstate(over="ignore"):
        cand = cand[_bucket(cand, n_buckets) == 0]
        grp, tag = _p2_group_tag(cand)
    pair = grp * np.uint64(32) + tag
    vals, counts = np.unique(pair, return_counts=True)
    best = vals[np.argmax(counts)]
    assert counts.max() >= n_tag
    g = best // np.uint64(32)
    same_tag = cand[pair == best][:n_tag]
    other = cand[(grp == g) & (pair != best)][: n_group - n_tag]
    assert len(other) == n_group - n_tag
    return np.concatenate([same_tag, other])


def test_keys_that_overflow_one_table_group_and_share_its_tags(G):
    from arroyo_b200 import ffi
    expected_keys = 4096
    n_buckets = -(-expected_keys // 1024)  # bdict.cuh: bd_buckets_for
    hot = colliding_keys(n_buckets)
    rng = np.random.default_rng(21)
    batches = gen_stream(rng, 400_000, 1_000, rate_per_s=20_000, batch=65_536)
    out = []
    for b in batches:
        key = b["key"].copy()
        pick = rng.random(len(key)) < 0.05  # few enough that bucket 0 stays within its partition regions
        key[pick] = hot[rng.integers(0, len(hot), int(pick.sum()))]
        out.append(O.Batch({"key": key, "value": b["value"], O.TIMESTAMP: b[O.TIMESTAMP]}))
    cfg = O.WindowAggConfig(width=4 * S, slide=S, key_names=["key"], aggs=SUM_AVG, window_index=1)
    want, got, gop = run_both(G, lambda: O.SlidingAggregatingWindowFunc(cfg),
                              lambda: G.SlidingAggregatingWindowFunc(cfg, flags=ffi.FLAG_TWO_PASS_ALWAYS,
                                                                     expected_keys=expected_keys), out)
    assert_same(want, got, float_cols=("avg",))
    assert set(hot.tolist()) <= {r["key"] for b in got for r in b.rows()}
    assert gop.stats()["rows_in"] == 400_000


def _device_run(pieces, n):
    """Tumbling 1 s SUM + COUNT over one pane of `n` device rows: the first 1000 rows, then the (first row, rows)
    slices `pieces` of the same columns in one call; the emitted window is compared with a group-by."""
    import pyarrow as pa
    import torch

    import arroyo_b200 as ab
    from arroyo_b200 import ffi, operators as native
    from arroyo_b200.multi_gpu import _Ptr

    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    torch.cuda.set_stream(torch.cuda.Stream(device=device))
    g = torch.Generator(device=device)
    g.manual_seed(7)
    ids = torch.randint(0, 50_000, (n,), generator=g, device=device, dtype=torch.int64)
    key = ids * 0x1E3779B97F4A7C15 % (1 << 62) - (1 << 61)
    val = torch.randint(-(1 << 31), 1 << 31, (n,), generator=g, device=device, dtype=torch.int64)
    ts = T0 + torch.randint(0, S, (n,), generator=g, device=device, dtype=torch.int64)
    cfg = ab.WindowAggConfig(width=S, key_names=["key"], aggs=[ab.Agg("sum", "value", "sum"), ab.Agg("count", None, "n")],
                             window_index=1)
    schema = pa.schema([("key", pa.int64()), ("value", pa.int64()), ("_timestamp", pa.timestamp("ns"))])
    op = native.TumblingAggregatingWindowFunc(cfg, input_schema=schema, device=0,
                                              stream=torch.cuda.current_stream().cuda_stream,
                                              flags=ffi.FLAG_TWO_PASS_ALWAYS, expected_keys=50_000)
    # a first small batch tells the operator where the stream is (the two passes need a known newest pane)
    first = 1000
    op.process_device_batch([key.data_ptr(), val.data_ptr(), ts.data_ptr()], first)
    op.flush()
    cols = (C.c_uint64 * (3 * len(pieces)))()
    rows = (C.c_int64 * len(pieces))()
    covered = first
    for i, (r0, nr) in enumerate(pieces):
        assert r0 == covered
        covered += nr
        for c, t in enumerate((key, val, ts)):
            cols[3 * i + c] = t.data_ptr() + 8 * r0
        rows[i] = nr
    assert covered == n
    op.process_device_batches(cols, rows, 3)
    got = None
    for nrow, ptrs in op.handle_watermark_device(T0 + 2 * S):
        assert got is None
        got = [torch.as_tensor(_Ptr(c, nrow), device=device).clone() for c in ptrs]
    st = op.stats()
    op.close()
    assert got is not None and st["rows_in"] == n
    uk, inv = torch.unique(key, return_inverse=True)
    want_sum = torch.zeros(uk.numel(), dtype=torch.int64, device=device).index_add_(0, inv, val)
    want_cnt = torch.zeros(uk.numel(), dtype=torch.int64, device=device).index_add_(0, inv, torch.ones_like(val))
    order = torch.argsort(got[0])
    assert torch.equal(got[0][order], uk)
    assert torch.equal(got[3][order], want_sum)
    assert torch.equal(got[4][order], want_cnt)


def test_sliced_device_batches_beside_aligned_ones():
    # after the first 1000 rows: 2^18 - 1001 rows from an aligned start (whole tiles by TMA, then a partial last tile),
    # 2^18 + 1 rows that start at an odd row (columns 8 bytes off 16-byte alignment), then 2^18 - 1 rows from an even
    # row again
    a = (1 << 18) - 1001
    b = (1 << 18) + 1
    c = (1 << 18) - 1
    assert (1000 + a) % 2 == 1 and (1000 + a + b) % 2 == 0
    _device_run([(1000, a), (1000 + a, b), (1000 + a + b, c)], 1000 + a + b + c)


def test_a_launch_whose_last_tile_is_partial():
    # one batch of 2^20 + 777 rows after the first 1000: every tile of it whole but the last
    n = 1000 + (1 << 20) + 777
    _device_run([(1000, n - 1000)], n)

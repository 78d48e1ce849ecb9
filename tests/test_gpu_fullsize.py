"""Parity at BASELINE.json's full sizes through size-independent properties (the oracle cannot run 288M rows in
seconds): checksums of checksums, row counts, sortedness, partition membership.  Sizes: config 2 and config 3 at the
full SF100 `store_sales` row count (287,997,024); config 4 at one GPU's share of the sort / shuffle (64M rows).
The expected values are computed with numpy directly on the generated columns, never through the engine."""
import os
import struct
import sys

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
import oracle
from auron_b200 import proto as P
from auron_b200 import runtime

pytestmark = pytest.mark.gpu

SF100 = bench.SF100_ROWS


def _run(plan, is_task_definition=False):
    td = plan if is_task_definition else P.task_definition(plan)
    with runtime.Task(td) as task:
        return pa.Table.from_batches(list(task), schema=task.schema)


def test_config2_full_size_checksums(tmp_path):
    # ParquetScan -> Filter -> HashAggregate over all 287,997,024 rows (SNAPPY pages), checked against numpy reductions of
    # the very arrays the files were written from (regenerated from the same seeds).  The files are written here, never taken
    # from a directory an earlier run left behind.
    files = bench.gen_dataset(str(tmp_path), SF100)
    paths = [f for f, _ in files]
    exp_cnt = exp_sum = 0
    seen = np.zeros(bench.N_ITEMS + 1, dtype=bool)
    cnt_g = np.zeros(bench.N_ITEMS + 1, dtype=np.int64)           # per group: COUNT(ss_quantity), SUM(ss_quantity)
    sum_g = np.zeros(bench.N_ITEMS + 1, dtype=np.int64)
    for i, (_, rows) in enumerate(files):
        rng = np.random.default_rng(42 + i)                       # same draws as bench.gen_file
        item = rng.integers(1, bench.N_ITEMS + 1, rows, dtype=np.int32)
        qty = rng.integers(1, 101, rows, dtype=np.int32)
        qnull = rng.random(rows) < 0.03
        date = rng.integers(bench.DATE_LO, bench.DATE_HI, rows, dtype=np.int32)
        dnull = rng.random(rows) < 0.04
        keep = (~dnull) & (date >= bench.FILTER_LO) & (date < bench.FILTER_HI)
        exp_cnt += int(np.count_nonzero(keep & ~qnull))
        exp_sum += int(qty[keep & ~qnull].astype(np.int64).sum())
        seen[item[keep]] = True
        sel = keep & ~qnull
        cnt_g += np.bincount(item[sel], minlength=bench.N_ITEMS + 1)
        sum_g += np.bincount(item[sel], weights=qty[sel].astype(np.float64), minlength=bench.N_ITEMS + 1).astype(np.int64)   # exact: < 2^53
    out = _run(bench.build_plan(P, paths, [os.path.getsize(p) for p in paths]), is_task_definition=True)
    for p in paths:                                                         # ~1.4 GB: not kept for pytest's retained temp dirs
        os.remove(p)
    assert out.num_rows == int(seen.sum())                                  # every selected item is a group, exactly once
    assert len(set(out.column(0).to_pylist())) == out.num_rows
    assert int(out.column(2).to_numpy().sum()) == exp_cnt                   # COUNT(ss_quantity)
    assert int(np.nansum(out.column(1).to_numpy(zero_copy_only=False).astype(np.float64))) == exp_sum   # SUM(ss_quantity) (exact in f64: < 2^53)
    # every group's own COUNT and SUM, not only their totals
    keys = out.column(0).to_numpy()
    assert np.array_equal(np.sort(keys), np.nonzero(seen)[0])
    assert np.array_equal(out.column(2).to_numpy(), cnt_g[keys])
    sums = out.column(1).combine_chunks()
    assert np.array_equal(np.asarray(sums.is_valid()), cnt_g[keys] > 0)         # SUM of no values is NULL (sum.rs:115)
    assert np.array_equal(sums.fill_null(0).to_numpy(), sum_g[keys])


def test_config3_full_size_join_counts():
    # store_sales (288M probe rows) JOIN date_dim (73,049 build rows): joined row count and two column checksums
    n = SF100
    rng = np.random.default_rng(7)
    date_lo = 2450816
    dkey = np.arange(2415022, 2415022 + 73049, dtype=np.int32)
    dyear = (1900 + np.arange(73049) // 365).astype(np.int32)
    dd = pa.table({"d_date_sk": pa.array(dkey), "d_year": pa.array(dyear)})
    chunk = 48_000_000
    exp_rows = exp_year = exp_qty = 0
    left = n
    while left > 0:
        m = min(chunk, left)
        sold = rng.integers(date_lo - 500, date_lo + 1826, m, dtype=np.int32)      # every key has exactly one date_dim row
        null = rng.random(m) < 0.04
        qty = rng.integers(1, 101, m, dtype=np.int32)
        runtime.put_device_batch("fs_ss", pa.record_batch({"ss_sold_date_sk": pa.array(sold, mask=null), "ss_quantity": pa.array(qty)}))
        ok = ~null
        exp_rows += int(ok.sum())
        exp_year += int(dyear[sold[ok] - 2415022].astype(np.int64).sum())
        exp_qty += int(qty[ok].astype(np.int64).sum())
        left -= m
    runtime.put_device_batch("fs_dd", dd.to_batches()[0])
    ss_schema = pa.schema([("ss_sold_date_sk", pa.int32()), ("ss_quantity", pa.int32())])
    try:
        j = P.hash_join(pa.schema(list(dd.schema) + list(ss_schema)), P.ffi_reader(dd.schema, "fs_dd"), P.ffi_reader(ss_schema, "fs_ss"),
                        [(P.col("d_date_sk"), P.col("ss_sold_date_sk"))], "INNER", "LEFT")
        plan = P.agg(j, [], [], [P.agg_expr("COUNT", [P.col("d_date_sk")], pa.int64()), P.agg_expr("SUM", [P.col("d_year")], pa.int64()),
                                 P.agg_expr("SUM", [P.col("ss_quantity")], pa.int64())], ["c", "y", "q"], ["PARTIAL"] * 3)
        out = _run(plan)
    finally:
        runtime.drop_device_resource("fs_ss")
        runtime.drop_device_resource("fs_dd")
    assert out.column(0).to_pylist() == [exp_rows]        # NULL keys never match (joins/test.rs null-key scenarios)
    assert out.column(1).to_pylist() == [exp_year]
    assert out.column(2).to_pylist() == [exp_qty]


def test_config4_sort_and_shuffle_64m(tmp_path):
    n = 64_000_000
    rng = np.random.default_rng(11)
    item = rng.integers(1, 204001, n, dtype=np.int32)
    ticket = rng.integers(1, 240_000_000, n, dtype=np.int64)
    t = pa.table({"ss_item_sk": pa.array(item), "ss_ticket_number": pa.array(ticket)})
    for b in t.to_batches(max_chunksize=16_000_000):
        runtime.put_device_batch("fs_t4", b)
    try:
        # SortExec: output is ordered, is a permutation of the input (checksums), and windows [offset, limit) agree with numpy
        srt = _run(P.sort(P.ffi_reader(t.schema, "fs_t4"), [P.sort_expr(P.col("ss_item_sk")), P.sort_expr(P.col("ss_ticket_number"))]))
        k = srt.column(0).to_numpy()
        v = srt.column(1).to_numpy()
        assert len(k) == n and bool(np.all(k[1:] >= k[:-1]))
        same = k[1:] == k[:-1]
        assert bool(np.all(v[1:][same] >= v[:-1][same]))                       # second key orders ties
        assert int(k.astype(np.int64).sum()) == int(item.astype(np.int64).sum()) and int(v.sum()) == int(ticket.sum())
        assert int(np.bitwise_xor.reduce(v)) == int(np.bitwise_xor.reduce(ticket))
        del srt, k, v
        # ShuffleWriterExec: every row lands in the partition Spark's murmur3 partitioner assigns it; nothing lost
        nparts = 200
        data, index = str(tmp_path / "s.data"), str(tmp_path / "s.index")
        _run(P.shuffle_writer(P.ffi_reader(t.schema, "fs_t4"), P.hash_repartition([P.col("ss_item_sk")], nparts), data, index))
    finally:
        runtime.drop_device_resource("fs_t4")
    offsets = struct.unpack(f"<{nparts + 1}q", open(index, "rb").read())
    assert offsets[0] == 0 and offsets[-1] == os.path.getsize(data)
    pid = oracle.partition_ids([pa.array(item)], nparts)
    exp_rows = np.bincount(pid, minlength=nparts)
    # exact per-partition sums of the int64 tickets: float64 bincount is exact on each 32-bit half (< 2^53)
    lo = np.bincount(pid, weights=(ticket & 0xFFFFFFFF).astype(np.float64), minlength=nparts)
    hi = np.bincount(pid, weights=(ticket >> 32).astype(np.float64), minlength=nparts)
    exp_sum = [(int(h) << 32) + int(l) for h, l in zip(hi, lo)]
    raw = open(data, "rb").read()
    total = 0
    for p in range(nparts):
        seg = raw[offsets[p]:offsets[p + 1]]
        pos, rows, tsum, bad = 0, 0, 0, 0
        while pos < len(seg):
            (blen,) = struct.unpack_from("<I", seg, pos)
            payload = pa.CompressedInputStream(pa.BufferReader(seg[pos + 4:pos + 4 + blen]), "lz4").read()
            pos += 4 + blen
            bpos = 0
            while bpos < len(payload):
                b, bpos = oracle.serde_read_batch(payload, t.schema, bpos)
                rows += b.num_rows
                tsum += int(b.column(1).to_numpy().sum())
                if p % 37 == 0:                                                 # membership re-checked on a sample of partitions
                    bad += int(np.count_nonzero(oracle.partition_ids([b.column(0)], nparts) != p))
        assert rows == exp_rows[p] and bad == 0, p
        assert tsum == exp_sum[p], p
        total += rows
    assert total == n

"""Pins the CPU oracle against the reference's own known-answer tests (SURVEY.md section 8c).

Every test names the reference test it reproduces (paths relative to the StarRocks tree).
"""
import os
import zlib

import numpy as np
import pytest

from starrocks_b200 import abi
from starrocks_b200.abi import Chunk

# known answers of the reference's hash functions and page codec (scripts/make_reference_vectors.py)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz")


# ---- be/test/exec/join_hash_map_test.cpp:924-1009  JoinKeyHash ---------------------------------
@pytest.mark.parametrize("width,stride,expect", [
    (32, 3, (0, 11)), (32, 7, (0, 14)), (32, 1, (4, 6)),
    (64, 3, (3, 7)), (64, 7, (4, 7)), (64, 1, (4, 6)),
])
def test_join_key_hash_bucket_occupancy(oracle, width, stride, expect):
    L = oracle.lib()
    num_buckets, log_buckets = 1 << 16, 16
    counts = np.zeros(num_buckets, dtype=np.int64)
    fn = L.orc_join_key_hash32 if width == 32 else L.orc_join_key_hash64
    for i in range(0, num_buckets * stride * 5, stride):
        counts[fn(i, log_buckets)] += 1
    assert (counts.min(), counts.max()) == expect


def test_join_key_hash_slice(oracle):
    # JoinKeyHash<Slice>()(Slice{"abcd",4}, 1<<16, 16) == 11538  (:1007-1008)
    buf = np.frombuffer(b"abcd", dtype=np.uint8).copy()
    assert oracle.lib().orc_join_key_hash_slice(buf.ctypes.data, 4, 1 << 16) == 11538


def test_calc_bucket_num(oracle):
    # CalcBucketNum / CalcBucketNums (:1012-1033)
    L = oracle.lib()
    assert L.orc_join_key_hash32(1, 2) == 2
    assert [L.orc_join_key_hash32(v, 2) for v in (1, 2, 3, 4)] == [2, 0, 3, 1]


def test_calc_bucket_size(oracle):
    # JoinBuildProbeFunc uses bucket_size 16 for row_count 10 (:1147-1150); helper :70-77
    L = oracle.lib()
    assert L.orc_calc_bucket_size(11) == 16
    assert L.orc_calc_bucket_size(1) == 2
    assert L.orc_calc_bucket_size(600001) == 1 << 20


# ---- be/test/base/hash/hash_util_test.cpp:78-100 ------------------------------------------------
def test_hash_util_goldens(oracle):
    L = oracle.lib()
    hello = np.frombuffer(b"hello", dtype=np.uint8).copy()
    assert L.orc_fnv_hash(hello.ctypes.data, 5, 0) == 0x1840de38
    assert L.orc_fnv_hash(hello.ctypes.data, 5, 0x811C9DC5) == 0x4f9f2cab
    assert L.orc_fnv_hash(hello.ctypes.data, 0, 0x811C9DC5) == 0x811C9DC5
    assert L.orc_xorshift32(1) == 0x00042021
    assert L.orc_xorshift32(0x12345678) == 0x87985aa5
    sr = np.frombuffer(b"starrocks", dtype=np.uint8).copy()
    assert L.orc_zlib_crc32(sr.ctypes.data, 9, 0) == zlib.crc32(b"starrocks", 0)
    # ReduceOp (hash_util.hpp:242-244)
    assert L.orc_reduce_op(0xFFFFFFFF, 8) == 7 and L.orc_reduce_op(0, 8) == 0
    assert L.orc_reduce_op(0x80000000, 3) == 1


# ---- be/test/column/column_filter_range_test.cpp:25-70 -----------------------------------------
def test_filter_range_goldens(oracle):
    L = oracle.lib()
    v = np.array([10, 11, 12, 13, 14, 15], dtype=np.int32)
    f = np.array([1, 0, 1, 0, 1, 0], dtype=np.uint8)
    assert L.orc_filter_range(f.ctypes.data, v.ctypes.data, 4, 0, 6) == 3
    assert list(v[:3]) == [10, 12, 14]
    d = np.array([0.1, 0.2, 0.3, 0.4, 0.5, 0.6], dtype=np.float64)
    f = np.array([1, 0, 1, 1, 0, 1], dtype=np.uint8)
    assert L.orc_filter_range(f.ctypes.data, d.ctypes.data, 8, 1, 5) == 3
    assert list(d[:3]) == [0.1, 0.3, 0.4]
    z = np.array([7, 8, 9, 10], dtype=np.int32)
    f0 = np.zeros(4, dtype=np.uint8)
    assert L.orc_filter_range(f0.ctypes.data, z.ctypes.data, 4, 0, 4) == 0
    o = np.array([100, 200, 300, 400, 500], dtype=np.int32)
    f1 = np.ones(5, dtype=np.uint8)
    assert L.orc_filter_range(f1.ctypes.data, o.ctypes.data, 4, 2, 5) == 5
    assert list(o) == [100, 200, 300, 400, 500]


# ---- join build / probe -------------------------------------------------------------------------
def _int_join(oracle, join_type=abi.JOIN_INNER, key_type=abi.TYPE_INT, build_out=(), probe_out=(), **kw):
    d = abi.make_join_desc(join_type, [1], [0], [key_type], build_out=build_out, probe_out=probe_out)
    return oracle.Join(d, **kw)


def _nullable_int32(count, start):
    # JoinHashMapTest::create_int32_nullable_column (:695-709): odd values are NULL
    vals = np.arange(start, start + count, dtype=np.int32)
    nulls = (vals % 2 != 0).astype(np.uint8)
    data = np.where(nulls == 1, 0, vals).astype(np.int32)
    return data, nulls


@pytest.mark.parametrize("method", ["BUCKET_CHAINED", "LINEAR_CHAINED", "RANGE_DIRECT_MAPPING",
                                    "DENSE_RANGE_DIRECT_MAPPING"])
def test_join_build_probe_func(oracle, method):
    # JoinBuildProbeFunc (:1138-1185): build {0..9}, probe {0..9}: every probe row finds exactly one
    j = _int_join(oracle, force_method=getattr(oracle, method))
    j.append_build(Chunk([(1, np.arange(10, dtype=np.int32), None)]))
    j.build()
    if method == "BUCKET_CHAINED":
        assert j.bucket_size == 16
    first, nxt = j.first(), j.next()
    probe = Chunk([(0, np.arange(10, dtype=np.int32), None)])
    pi, bi, res = j.probe_chunk(probe)
    assert res.count == 10 and not res.has_remain
    assert list(pi) == list(range(10))
    assert list(bi) == [i + 1 for i in range(10)]  # build row index is 1-based (row 0 = sentinel)
    assert res.match_flag == 1  # ALL_MATCH_ONE
    assert nxt[0] == 0 and len(first) > 0


@pytest.mark.parametrize("method", ["BUCKET_CHAINED", "LINEAR_CHAINED", "RANGE_DIRECT_MAPPING"])
def test_join_build_probe_func_nullable(oracle, method):
    # JoinBuildProbeFuncNullable (:1188-1240): odd rows are NULL on both sides -> found 0 times
    j = _int_join(oracle, force_method=getattr(oracle, method))
    bd, bn = _nullable_int32(10, 0)
    j.append_build(Chunk([(1, bd, bn)]))
    j.build()
    pd, pn = _nullable_int32(10, 0)
    pi, bi, res = j.probe_chunk(Chunk([(0, pd, pn)]))
    assert list(pi) == [0, 2, 4, 6, 8]
    assert list(bi) == [1, 3, 5, 7, 9]


def test_direct_mapping_join_build_probe_func(oracle):
    # DirectMappingJoinBuildProbeFunc (:1243-1289): TINYINT keys -> DIRECT_MAPPING
    j = _int_join(oracle, key_type=abi.TYPE_TINYINT, build_out=[1], probe_out=[0])
    j.append_build(Chunk([(1, np.array([-5, -3, -1, 0, 1, 3, 5], dtype=np.int8), None)]))
    j.build()
    assert j.method == oracle.DIRECT_MAPPING and j.bucket_size == 256
    probe = Chunk([(0, np.array([-8, -5, 0, 1, 2, 3, 4, 5], dtype=np.int8), None)])
    pi, bi = j.probe_all(probe)
    out = j.output(probe, pi, bi)
    assert [s for s, _, _ in out] == [0, 1]
    assert sorted(out[1][1].tolist()) == [-5, 0, 1, 3, 5]


def test_direct_mapping_join_build_probe_func_nullable(oracle):
    # DirectMappingJoinBuildProbeFuncNullable (:1292-1351)
    j = _int_join(oracle, key_type=abi.TYPE_TINYINT, build_out=[1], probe_out=[0])
    j.append_build(Chunk([(1, np.array([-5, 0, 0, 0, 1, 3, 5], dtype=np.int8),
                           np.array([0, 1, 0, 1, 0, 0, 0], dtype=np.uint8))]))
    j.build()
    probe = Chunk([(0, np.array([-5, 0, 0, 0, 3, 0, 5, 0], dtype=np.int8),
                    np.array([0, 1, 0, 1, 0, 1, 0, 1], dtype=np.uint8))])
    pi, bi = j.probe_all(probe)
    out = j.output(probe, pi, bi)
    assert sorted(out[1][1].tolist()) == [-5, 0, 3, 5]
    assert out[1][2].tolist() == [0, 0, 0, 0]


def test_probe_from_ht_first_one_to_one_all_match(oracle):
    # ProbeFromHtFirstOneToOneAllMatch (:1656-1695)
    j = _int_join(oracle)
    j.append_build(Chunk([(1, np.arange(4096, dtype=np.int32), None)]))
    j.build()
    pi, bi, res = j.probe_chunk(Chunk([(0, np.arange(4096, dtype=np.int32), None)]))
    assert res.match_flag == 1 and not res.has_remain and res.cur_probe_index == 0
    assert res.count == 4096 and res.cur_row_match_count == 0
    assert np.array_equal(pi, np.arange(4096)) and np.array_equal(bi, np.arange(4096) + 1)


def test_probe_from_ht_first_one_to_one_most_match(oracle):
    # ProbeFromHtFirstOneToOneMostMatch (:1698-1745): a quarter of the probe rows find no equal key
    j = _int_join(oracle)
    keys = np.array([i for i in range(4096) if i % 4 != 0], dtype=np.int32)
    j.append_build(Chunk([(1, keys, None)]))
    j.build()
    pi, bi, res = j.probe_chunk(Chunk([(0, np.arange(4096, dtype=np.int32), None)]))
    assert res.match_flag == 2 and not res.has_remain and res.count == 3072
    assert np.array_equal(pi, keys.astype(np.uint32))


@pytest.mark.parametrize("method", ["RANGE_DIRECT_MAPPING", "BUCKET_CHAINED", "LINEAR_CHAINED"])
def test_probe_from_ht_first_one_to_many(oracle, method):
    # ProbeFromHtFirstOneToMany (:1748-1812): 3000 probe rows x 2 build matches, chunk_size 4096
    j = _int_join(oracle, force_method=getattr(oracle, method))
    build = np.concatenate([np.arange(4096), np.arange(4096)]).astype(np.int32)
    j.append_build(Chunk([(1, build, None)]))
    j.build()
    if method == "RANGE_DIRECT_MAPPING":
        # same chains the reference test builds by hand: head = second copy, next -> first copy
        assert np.array_equal(j.next()[4097:], np.arange(1, 4097))
        assert not j.next()[1:4097].any()
    probe = Chunk([(0, np.arange(3000, dtype=np.int32), None)])
    pi1, bi1, r1 = j.probe_chunk(probe, True)
    assert r1.match_flag == 0 and r1.has_remain and r1.count == 4096
    assert r1.cur_probe_index == 2048 and r1.cur_row_match_count == 1
    pi2, bi2, r2 = j.probe_chunk(probe, False)
    assert r2.match_flag == 0 and not r2.has_remain and r2.count == 1904
    assert r2.cur_probe_index == 0 and r2.cur_row_match_count == 0
    pairs = sorted(zip(np.concatenate([pi1, pi2]).tolist(), np.concatenate([bi1, bi2]).tolist()))
    expect = sorted([(i, i + 1) for i in range(3000)] + [(i, 4097 + i) for i in range(3000)])
    assert pairs == expect


def test_probe_left_outer_found_empty(oracle):
    # ProbeFromHtForLeftJoinFoundEmpty (:1815-1880): probe rows without a match emit build_index 0
    j = _int_join(oracle, join_type=abi.JOIN_LEFT_OUTER)
    j.append_build(Chunk([(1, np.arange(0, 100, 2, dtype=np.int32), None)]))
    j.build()
    pi, bi, res = j.probe_chunk(Chunk([(0, np.arange(100, dtype=np.int32), None)]))
    assert res.count == 100 and list(pi) == list(range(100))
    assert all((b == 0) == (i % 2 == 1) for i, b in enumerate(bi))


def test_one_key_join_hash_table(oracle):
    # OneKeyJoinHashTable (:2042-2088): build {0..9},{10..19},{20..29}; probe {1..5},{11..},{21..}
    d = abi.make_join_desc(abi.JOIN_INNER, [3], [0], [abi.TYPE_INT], build_out=[3, 4, 5], probe_out=[0, 1, 2])
    j = oracle.Join(d)
    j.append_build(Chunk([(3 + k, np.arange(10 * k, 10 * k + 10, dtype=np.int32), None) for k in range(3)]))
    j.build()
    probe = Chunk([(k, np.arange(1 + 10 * k, 6 + 10 * k, dtype=np.int32), None) for k in range(3)])
    pi, bi = j.probe_all(probe)
    out = j.output(probe, pi, bi)
    assert len(out) == 6
    for k, (slot, data, _) in enumerate(out):
        assert slot == k
        assert data.tolist() == list(range(1 + 10 * (k % 3), 6 + 10 * (k % 3)))


def test_one_nullable_key_join_hash_table(oracle):
    # OneNullableKeyJoinHashTable (:2091-2140): NULL keys never match
    d = abi.make_join_desc(abi.JOIN_INNER, [3], [0], [abi.TYPE_INT], build_out=[3], probe_out=[0])
    j = oracle.Join(d)
    bd, bn = _nullable_int32(10, 0)
    j.append_build(Chunk([(3, bd, bn)]))
    j.build()
    pd, pn = _nullable_int32(5, 1)
    probe = Chunk([(0, pd, pn)])
    pi, bi = j.probe_all(probe)
    out = j.output(probe, pi, bi)
    assert out[0][1].tolist() == [2, 4] and out[1][1].tolist() == [2, 4]


def test_selector_rules(oracle):
    # JoinHashMapSelector::_determine_hash_map_method (join_hash_table.cpp:225-350)
    def method(keys, join_type=abi.JOIN_INNER, **kw):
        j = _int_join(oracle, join_type=join_type, **kw)
        j.append_build(Chunk([(1, np.asarray(keys, dtype=np.int32), None)]))
        j.build()
        return j.method
    assert method(np.arange(1, 1001)) == oracle.RANGE_DIRECT_MAPPING          # interval <= bucket_size
    assert method([1, 1 << 19]) == oracle.RANGE_DIRECT_MAPPING                 # interval <= L2
    assert method([1, 1 << 30]) == oracle.LINEAR_CHAINED                       # sparse -> linear chained
    assert method([1, 1 << 30], l2=1 << 31) == oracle.RANGE_DIRECT_MAPPING
    assert method(np.arange(1, 1001), join_type=abi.JOIN_LEFT_SEMI) == oracle.RANGE_DIRECT_MAPPING_SET
    # dense: interval/4 + rows*4 <= 1.1*bucket*4 but interval > bucket and > L2
    keys = np.arange(0, 3_000_000, 5, dtype=np.int32)
    assert method(keys, l2=1 << 20) == oracle.DENSE_RANGE_DIRECT_MAPPING


# ---- SQL goldens: test/sql/test_join/R/test_join_range_direct_mapping ---------------------------
def sql_golden_t1(n=1_280_000):
    """t1 of test/sql/test_join/T/test_join_range_direct_mapping: idx = row_number() = 1..n,
    c_int = idx, c_int_null = idx if idx % 13 == 0 else NULL, c_bigint_null on % 14."""
    idx = np.arange(1, n + 1, dtype=np.int32)
    null13 = (idx % 13 != 0).astype(np.uint8)
    null14 = (idx % 14 != 0).astype(np.uint8)
    return idx, null13, idx.astype(np.int64), null14


def test_sql_golden_range_direct_mapping_counts(oracle):
    # R/test_join_range_direct_mapping: `t1 JOIN t1 t2 on c_int` -> 1280000; on c_int_null -> 98461;
    # `LEFT JOIN on c_bigint_null` -> 1280000 rows of which 91428 have a build match;
    # w1 = t1 union all t1 self-joined on c_int -> 5120000
    idx, null13, big, null14 = sql_golden_t1()
    for key_nulls, expect in ((None, 1280000), (null13, 98461)):
        j = _int_join(oracle)
        j.append_build(Chunk([(1, idx, key_nulls)]))
        j.build()
        assert j.method == oracle.RANGE_DIRECT_MAPPING
        pi, bi = j.probe_all(Chunk([(0, idx, key_nulls)]))
        assert len(pi) == expect
    j = _int_join(oracle, join_type=abi.JOIN_LEFT_OUTER, key_type=abi.TYPE_BIGINT)
    j.append_build(Chunk([(1, big, null14)]))
    j.build()
    pi, bi = j.probe_all(Chunk([(0, big, null14)]))
    assert len(pi) == 1280000 and int((bi != 0).sum()) == 91428
    # `where t2.c_int % 10 != 0` on the joined rows -> 73143
    t2_c_int = idx[np.maximum(bi, 1) - 1]
    assert int(((bi != 0) & (t2_c_int % 10 != 0)).sum()) == 73143
    w1 = np.concatenate([idx, idx])
    j = _int_join(oracle)
    j.append_build(Chunk([(1, w1, None)]))
    j.build()
    pi, bi = j.probe_all(Chunk([(0, w1, None)]), cap=5_200_000)
    assert len(pi) == 5120000


# ---- aggregate: be/test/exprs/agg/aggregate_test.cpp:61-83 test_sum -----------------------------
@pytest.mark.parametrize("typ,np_t", [(abi.TYPE_SMALLINT, np.int16), (abi.TYPE_INT, np.int32),
                                      (abi.TYPE_BIGINT, np.int64), (abi.TYPE_FLOAT, np.float32),
                                      (abi.TYPE_DOUBLE, np.float64)])
def test_sum_goldens(oracle, typ, np_t):
    col1 = np.array(list(range(1024)) + [100, 200], dtype=np_t)   # gen_input_column1
    col2 = np.arange(2000, 3000, dtype=np_t)                      # gen_input_column2
    d = abi.make_agg_desc(fns=[(abi.AGG_SUM, typ, 10, [("col", 0)])])
    a1, a2 = oracle.Agg(d), oracle.Agg(d)
    a1.push(Chunk([(0, col1, None)]))
    a2.push(Chunk([(0, col2, None)]))
    assert a1.output()[0][1][0] == 524076
    assert a2.output()[0][1][0] == 2499500
    a2.merge(a1)
    assert a2.output()[0][1][0] == 3023576


def test_count_avg_minmax_goldens(oracle):
    # aggregate_test.cpp test_count / test_avg / test_max / test_min over the same generators
    col1 = np.array(list(range(1024)) + [100, 200], dtype=np.int32)
    fns = [(abi.AGG_COUNT, abi.TYPE_INT, 10, [("col", 0)]), (abi.AGG_AVG, abi.TYPE_INT, 11, [("col", 0)]),
           (abi.AGG_MAX, abi.TYPE_INT, 12, [("col", 0)]), (abi.AGG_MIN, abi.TYPE_INT, 13, [("col", 0)]),
           (abi.AGG_COUNT_STAR, abi.TYPE_INT, 14, None)]
    a = oracle.Agg(abi.make_agg_desc(fns=fns))
    a.push(Chunk([(0, col1, None)]))
    out = a.output()
    assert out[0][1][0] == 1026
    assert out[1][1][0] == pytest.approx(524076 / 1026)
    assert out[2][1][0] == 1023 and out[3][1][0] == 0 and out[4][1][0] == 1026


@pytest.mark.parametrize("typ,dt", [(abi.TYPE_SMALLINT, np.int16), (abi.TYPE_INT, np.int32), (abi.TYPE_BIGINT, np.int64)])
def test_count_distinct_goldens(oracle, typ, dt):
    # aggregate_test.cpp:752-760 test_count_distinct: multi_distinct_count over gen_input_column1 (0..1023, 100, 200) = 1024,
    # over gen_input_column2 (2000..2999) = 1000, merged = 2024 (base_aggregate_test.h:83-112,203-237)
    col1 = np.array(list(range(1024)) + [100, 200], dtype=dt)
    col2 = np.arange(2000, 3000, dtype=dt)
    d = abi.make_agg_desc(fns=[(abi.AGG_COUNT_DISTINCT, typ, 10, [("col", 0)])])
    a, b = oracle.Agg(d), oracle.Agg(d)
    a.push(Chunk([(0, col1, None)]))
    b.push(Chunk([(0, col2, None)]))
    assert a.output()[0][1][0] == 1024
    assert b.output()[0][1][0] == 1000
    b.merge(a)
    assert b.output()[0][1][0] == 2024
    # grouped, with NULL inputs: NULLs are not counted, an all-NULL group reports 0
    g = np.array([0, 0, 0, 1, 1, 2], dtype=np.int32)
    v = np.array([5, 5, 7, 9, 9, 4], dtype=dt)
    nl = np.array([0, 0, 0, 0, 1, 1], dtype=np.uint8)
    c = oracle.Agg(abi.make_agg_desc([1], [abi.TYPE_INT], fns=[(abi.AGG_COUNT_DISTINCT, typ, 10, [("col", 0)])]))
    c.push(Chunk([(0, v, nl), (1, g, None)]))
    out = c.output()
    assert sorted(zip(out[0][1].tolist(), out[1][1].tolist())) == [(0, 2), (1, 1), (2, 0)]


def test_sum_nullable_all_null_is_null(oracle):
    # test_sum_nullable (aggregate_test.cpp:962): NULL inputs are skipped, all-NULL -> NULL result
    d = abi.make_agg_desc(fns=[(abi.AGG_SUM, abi.TYPE_INT, 10, [("col", 0)])])
    a = oracle.Agg(d)
    a.push(Chunk([(0, np.arange(100, dtype=np.int32), (np.arange(100) % 2).astype(np.uint8))]))
    assert a.output()[0][1][0] == sum(range(0, 100, 2)) and a.output()[0][2][0] == 0
    b = oracle.Agg(d)
    b.push(Chunk([(0, np.arange(10, dtype=np.int32), np.ones(10, dtype=np.uint8))]))
    assert b.output()[0][2][0] == 1


# ---- test/sql/test_exchange_hash_function: sum/count per c0 % 10 bucket ------------------------
def test_group_by_golden_mod10(oracle):
    # c0 = 1..1000 grouped by c0 % 10: (0,100,50500), (1,100,49600), ...
    c0 = np.arange(1, 1001, dtype=np.int32)
    d = abi.make_agg_desc([1], [abi.TYPE_INT], fns=[(abi.AGG_COUNT_STAR, abi.TYPE_INT, 10, None),
                                                     (abi.AGG_SUM, abi.TYPE_INT, 11, [("col", 0)])])
    a = oracle.Agg(d)
    a.push(Chunk([(0, c0, None), (1, (c0 % 10).astype(np.int32), None)]))
    out = a.output()
    rows = sorted(zip(out[0][1].tolist(), out[1][1].tolist(), out[2][1].tolist()))
    assert rows[0] == (0, 100, 50500) and rows[1] == (1, 100, 49600)
    assert [r[0] for r in rows] == list(range(10))
    # insertion order of the state arena (aggregator.cpp:1718-1724): first seen key first
    assert out[0][1].tolist() == [1, 2, 3, 4, 5, 6, 7, 8, 9, 0]


# ---- exchange partition -------------------------------------------------------------------------
def test_hash_partition_matches_python_fnv(oracle):
    vals = np.array([0, 1, 2, 1000, -1, 123456789], dtype=np.int32)

    def fnv(b, h):
        for x in b:
            h = ((x ^ h) * 0x01000193) & 0xFFFFFFFF
        return h
    d = abi.make_part_desc([0], 8)
    hv, ch, ri, st = oracle.hash_partition(d, Chunk([(0, vals, None)]))
    exp = [fnv(int(v).to_bytes(4, "little", signed=True), 0x811C9DC5) for v in vals]
    assert hv.tolist() == exp
    assert ch.tolist() == [(h * 8) >> 32 for h in exp]
    # stable counting sort: rows of each channel in input order
    assert sorted(ri.tolist()) == list(range(len(vals)))
    for c in range(8):
        rows = ri[st[c]:st[c + 1]].tolist()
        assert rows == sorted(rows) and all(ch[r] == c for r in rows)


# ---- runtime filter (be/test/runtime/runtime_filter_core_test.cpp) -------------------------------
def test_simd_block_filter_insert_and_test_golden(oracle):
    # :49-61 SimdBlockFilterInsertAndTest: init(100); insert_hash(1, 18, ..., 188); every inserted hash tests true,
    # hash + 1 tests false
    bf = oracle.RuntimeFilter(abi.TYPE_BIGINT, 100)
    assert bf.info().log_num_buckets == 2          # ceil(log2(100)) - 5 = 2 -> 4 buckets of 32 bytes
    for i in range(1, 201, 17):
        bf.insert_hash(i)
    for i in range(1, 201, 17):
        assert bf.test_hash(i) and not bf.test_hash(i + 1)
    # make_mask in plain Python: bit (uint32(hash >> log_buckets) * SALT[k]) >> 27 of word k of bucket hash & mask
    salt = [0x47b6137b, 0x44974d91, 0x8824ad5b, 0xa2b7289d, 0x705495c7, 0x2df1424b, 0x9efc4947, 0x5c6bfb31]
    exp = np.zeros(4 * 8, dtype=np.uint32)
    for i in range(1, 201, 17):
        for k in range(8):
            exp[8 * (i & 3) + k] |= np.uint32(1 << ((((i >> 2) * salt[k]) & 0xFFFFFFFF) >> 27))
    assert np.array_equal(bf.directory(), exp)


def test_simd_block_filter_merge_golden(oracle):
    # :79-102 SimdBlockFilterMerge
    left, right, merged = (oracle.RuntimeFilter(abi.TYPE_BIGINT, 100) for _ in range(3))
    for i in range(1, 201, 17):
        left.insert_hash(i)
        right.insert_hash(i + 1)
    merged.merge(left)
    merged.merge(right)
    for i in range(1, 201, 17):
        assert merged.test_hash(i) and merged.test_hash(i + 1) and not merged.test_hash(i + 2)


def test_min_max_runtime_filter_golden(oracle):
    # :104-123 MinMaxRangeAndNullableSemantics: insert 10, 20 -> {5,10,15,20,25} -> 0,1,1,1,0; NULL rows 0 until insert_null
    rf = oracle.RuntimeFilter(abi.TYPE_INT, 2, with_bloom=False)
    rf.insert(Chunk([(0, np.array([10, 20], dtype=np.int32), None)]), 0)
    col = np.array([5, 10, 15, 20, 25, 0, 0], dtype=np.int32)
    nulls = np.array([0, 0, 0, 0, 0, 1, 1], dtype=np.uint8)
    assert rf.evaluate(Chunk([(0, col[:5].copy(), None)]), 0).tolist() == [0, 1, 1, 1, 0]
    assert rf.evaluate(Chunk([(0, col, nulls)]), 0).tolist() == [0, 1, 1, 1, 0, 0, 0]
    rf.insert(Chunk([(0, np.array([0], dtype=np.int32), np.array([1], dtype=np.uint8))]), 0, insert_nulls=True)
    assert rf.evaluate(Chunk([(0, col, nulls)]), 0).tolist() == [0, 1, 1, 1, 0, 1, 1]


def test_runtime_bloom_filter_values(oracle):
    # RuntimeBloomFilter::compute_hash = phmap_mix<8>(std::hash<T>(v)) (runtime_filter.h:1270-1276, phmap_utils.h:86-95)
    def mix(a):
        p = (a & 0xFFFFFFFFFFFFFFFF) * 0xde5fb9d2630458e9
        return ((p >> 64) + p) & 0xFFFFFFFFFFFFFFFF
    for v in (0, 1, 42, -1, 2**31 - 1, -2**31, 123456789012345):
        assert oracle.value_hash(v) == mix(v)
    rng = np.random.default_rng(5)
    keys = rng.integers(-10**6, 10**6, 5000, dtype=np.int32)
    rf = oracle.RuntimeFilter(abi.TYPE_INT, len(keys))
    rf.insert(Chunk([(0, keys, None)]), 0)
    assert rf.evaluate(Chunk([(0, keys, None)]), 0).all()                      # no false negatives
    other = rng.integers(2 * 10**6, 3 * 10**6, 5000, dtype=np.int32)
    assert not rf.evaluate(Chunk([(0, other, None)]), 0).any()                 # outside [min, max]
    inside = np.setdiff1d(np.arange(-10**6, 10**6, 7, dtype=np.int32), keys)[:20000]
    fp = rf.evaluate(Chunk([(0, inside, None)]), 0).mean()
    assert fp < 0.05                                                           # 8 bits per key, 8 probes in one block


def _rf_reference_evaluate_vectors(make_filter):
    """runtime_filter_core_test.cpp:125-163 RuntimeBloomFilterEvaluateConstAndNullableColumns and :227-263
    RuntimeFilterBuilderFill{OnNullableColumn,WithEqNull}: known answers of evaluate() on const / NULL / nullable columns.
    `make_filter(expected_rows)` -> object with insert(chunk, slot, insert_nulls) / evaluate(chunk, slot)."""
    i32 = lambda xs: np.array(xs, dtype=np.int32)  # noqa: E731
    rf = make_filter(100)
    rf.insert(Chunk([(0, i32([10, 20]), None)]), 0)
    assert rf.evaluate(Chunk([(0, i32([10] * 8), None)]), 0).tolist() == [1] * 8           # const hit
    assert rf.evaluate(Chunk([(0, i32([11] * 8), None)]), 0).tolist() == [0] * 8           # const miss INSIDE [min, max]: the bloom part
    all_null = Chunk([(0, i32([0] * 8), np.ones(8, dtype=np.uint8))])
    assert rf.evaluate(all_null, 0).tolist() == [0] * 8                                    # const NULL, filter has no NULL
    nullable = Chunk([(0, i32([10, 11, 20, 21, 0, 0]), np.array([0, 0, 0, 0, 1, 1], dtype=np.uint8))])
    assert rf.evaluate(nullable, 0).tolist() == [1, 0, 1, 0, 0, 0]
    rf.insert(Chunk([(0, i32([0]), np.ones(1, dtype=np.uint8))]), 0, insert_nulls=True)   # insert_null()
    assert rf.evaluate(all_null, 0).tolist() == [1] * 8
    assert rf.evaluate(nullable, 0).tolist() == [1, 0, 1, 0, 1, 1]
    # RuntimeFilterBuilder::fill on a nullable column: eq_null = false skips the NULL, eq_null = true records it
    build = Chunk([(0, i32([10, 20, 0]), np.array([0, 0, 1], dtype=np.uint8))])
    plain, eq_null = make_filter(64), make_filter(64)
    plain.insert(build, 0, insert_nulls=False)
    eq_null.insert(build, 0, insert_nulls=True)
    assert plain.info().has_null == 0 and eq_null.info().has_null == 1
    assert plain.evaluate(Chunk([(0, i32([10, 20]), None)]), 0).tolist() == [1, 1]
    three_nulls = Chunk([(0, i32([0, 0, 0]), np.ones(3, dtype=np.uint8))])
    assert eq_null.evaluate(three_nulls, 0).tolist() == [1, 1, 1]
    assert plain.evaluate(three_nulls, 0).tolist() == [0, 0, 0]


def test_runtime_bloom_filter_evaluate_and_fill_golden(oracle):
    _rf_reference_evaluate_vectors(lambda n: oracle.RuntimeFilter(abi.TYPE_INT, n))


# ---- test/sql/test_agg/R/test_agg_compressed_key: the compressed-key (range-declared) aggregator on nullable keys -------
def _compressed_key_table():
    """all_t0 of the SQL test, integer columns only: x = 1..30000; c1 tinyint = x % 200 (128..199 overflow the TINYINT and
    load as NULL, which is what the goldens show), c2 smallint / c3 int / c4 bigint = x % 200, c13 tinyint / c14 smallint
    = x % 8, c15 int = x % 16, c16 bigint = x % 200 (NOT NULL columns), plus the two literal rows."""
    x = np.arange(1, 30001)
    m = x % 200
    c1, c1n = np.where(m < 128, m, 0), (m >= 128).astype(np.uint8)
    cols = {1: (np.concatenate([c1, [0, -1]]).astype(np.int8), np.concatenate([c1n, [1, 0]]).astype(np.uint8), abi.TYPE_TINYINT),
            2: (np.concatenate([m, [0, -2]]).astype(np.int16), np.array([0] * 30000 + [1, 0], dtype=np.uint8), abi.TYPE_SMALLINT),
            3: (np.concatenate([m, [0, -3]]).astype(np.int32), np.array([0] * 30000 + [1, 0], dtype=np.uint8), abi.TYPE_INT),
            4: (np.concatenate([m, [0, 0]]).astype(np.int64), np.array([0] * 30000 + [1, 1], dtype=np.uint8), abi.TYPE_BIGINT),
            13: (np.concatenate([x % 8, [-1, -1]]).astype(np.int8), None, abi.TYPE_TINYINT),
            14: (np.concatenate([x % 8, [-2, -2]]).astype(np.int16), None, abi.TYPE_SMALLINT),
            16: (np.concatenate([m, [-4, -4]]).astype(np.int64), None, abi.TYPE_BIGINT)}
    return cols


COMPRESSED_KEY_RANGES = {1: (-1, 127), 2: (-2, 199), 3: (-3, 199), 4: (0, 199), 13: (-1, 7), 14: (-2, 7), 16: (-4, 199)}
# (group-by columns) -> {position in ORDER BY keys ASC NULLS FIRST: expected row}; "last" = ORDER BY keys DESC LIMIT 1
COMPRESSED_KEY_GOLDENS = [
    ((1,), {0: (None, None), 1: (-1, -1), 2: (0, 0)}),                                   # :159-164
    ((1, 2), {0: (None, None, None), 1: (None, 128, None), 2: (None, 129, None)}),       # :165-170
    ((2,), {3: (1, 150), "last": (199, None)}), ((3,), {3: (1, 150), "last": (199, None)}),
    ((4,), {3: (2, 300), "last": (199, None)}), ((13,), {3: (2, 148800), "last": (7, 160800)}),
    ((14,), {3: (2, 148800), "last": (7, 160800)}), ((16,), {3: (2, 300), "last": (199, None)}),
    ((3, 4), {30: (28, 28, 4200)}),                                                       # :262-265
]


def _compressed_key_check(run_agg):
    """run_agg(desc, chunk) -> sorted rows (None first).  Every query is SUM(c1) GROUP BY the listed columns with the
    min/max statistics the FE would pass (the compressed-key variants, aggregator.cpp:1516-1566)."""
    cols = _compressed_key_table()
    for keys, expect in COMPRESSED_KEY_GOLDENS:
        d = abi.make_agg_desc(list(keys), [cols[k][2] for k in keys], fns=[(abi.AGG_SUM, abi.TYPE_TINYINT, 100, [("col", 1)])],
                              ranges=[COMPRESSED_KEY_RANGES[k] for k in keys], group_nullable=[1 if cols[k][1] is not None else 0 for k in keys])
        need = sorted(set(keys) | {1})
        rows = run_agg(d, Chunk([(k, cols[k][0], cols[k][1], cols[k][2]) for k in need]))
        for pos, want in expect.items():
            assert rows[-1 if pos == "last" else pos] == want, (keys, pos)


def test_agg_compressed_key_sql_goldens(oracle):
    from tests.helpers import oracle_rows

    def run(d, chunk):
        a = oracle.Agg(d)
        a.push(chunk)
        return oracle_rows(a)
    _compressed_key_check(run)


def test_divide_by_zero_is_null(oracle):
    # VectorizedDiv runs under ArithmeticRightZeroCheck (be/src/exprs/arithmetic_operation.h:638): x / 0 is NULL, for
    # DOUBLE as well as for integers cast to DOUBLE; SUM / COUNT over the quotient skip those rows
    a = np.array([6, 7, 8, 9], dtype=np.int64)
    b = np.array([3, 0, 2, 0], dtype=np.int64)
    vals, nul = oracle.eval_expr(abi.make_expr([("col", 0), ("col", 1), "/"]), Chunk([(0, a, None), (1, b, None)]))
    assert nul.tolist() == [0, 1, 0, 1]
    assert vals[0] == 2.0 and vals[2] == 4.0
    x = np.array([1.5, -2.0, 0.0], dtype=np.float64)
    y = np.array([0.0, 0.5, 0.0], dtype=np.float64)
    vals, nul = oracle.eval_expr(abi.make_expr([("col", 0), ("col", 1), "/"]), Chunk([(0, x, None), (1, y, None)]))
    assert nul.tolist() == [1, 0, 1] and vals[1] == -4.0
    d = abi.make_agg_desc(fns=[(abi.AGG_SUM, abi.TYPE_DOUBLE, 10, [("col", 0), ("col", 1), "/"]),
                               (abi.AGG_COUNT, abi.TYPE_DOUBLE, 11, [("col", 0), ("col", 1), "/"])])
    ag = oracle.Agg(d)
    ag.push(Chunk([(0, a, None), (1, b, None)]))
    out = ag.output()
    assert out[0][1][0] == 6.0 and out[1][1][0] == 2          # 6/3 + 8/2, two non-NULL quotients


def test_xxh3_64_reference_goldens(oracle):
    # HashFunctionsTest.test_xx_hash3_64 (be/test/exprs/hash_functions_test.cpp:85-118): xx_hash3_64('hello') and
    # ('starrocks') with XXHASH3_64_SEED = 0; two columns chain the first hash as the seed of the second.  5 bytes take
    # XXH3_len_4to8_64b, 9 bytes XXH3_len_9to16_64b.
    L = oracle.lib()

    def h(b, seed):
        buf = np.frombuffer(b, dtype=np.uint8).copy()
        v = L.orc_xxh3_64(buf.ctypes.data, len(b), seed)
        return v - (1 << 64) if v >= 1 << 63 else v
    assert h(b"hello", 0) == -7685981735718036227
    assert h(b"starrocks", 0) == 6573472450560322992
    assert h(b"world", h(b"hello", 0) & ((1 << 64) - 1)) == 7001965798170371843
    assert h(b"starrocks", h(b"hello", 0) & ((1 << 64) - 1)) == 2803320466222626098


def test_xxh3_64_against_the_reference_header(oracle):
    # every length 1..16, 200 random byte strings each, random 64-bit and 32-bit seeds (the exchange feeds 32-bit seeds):
    # the restatement against the hashes of the xxHash library the reference vendors (tests/golden, written by
    # scripts/make_reference_vectors.py), and -- where `make -C oracle ref` built oracle/_ref/libxxh3_ref.so from the
    # reference's own xxhash.h -- the reference header against the same hashes
    g = np.load(GOLDEN)
    ref = oracle.ref_xxh3()
    fns = [oracle.lib().orc_xxh3_64] + ([ref.ref_xx_hash3_64] if ref is not None else [])
    for buf, n, seed, want in zip(g["xxh3_data"], g["xxh3_len"].tolist(), g["xxh3_seed"].tolist(), g["xxh3_hash"].tolist()):
        buf = np.ascontiguousarray(buf)
        for fn in fns:
            assert fn(buf.ctypes.data, n, seed) == want, (fn.__name__, n, seed)


def test_hash_partition_xxh3_matches_value_hash(oracle):
    # exchange_hash_function_version = 1: per partition column hash = (uint32) xx_hash3_64(value, width, seed = hash so far),
    # from XXH3_SEED_32 = 0x9E3779B1 (exchange_sink_operator.cpp:597-601); channel = ReduceOp(hash, n)
    rng = np.random.default_rng(12)
    a = rng.integers(-10**9, 10**9, 1000, dtype=np.int32)
    b = rng.integers(-10**15, 10**15, 1000, dtype=np.int64)
    d = abi.make_part_desc([0, 1], 7, hash_fn=abi.HASH_XXH3)
    hv, ch, ri, st = oracle.hash_partition(d, Chunk([(0, a, None), (1, b, None)]))
    L = oracle.lib()
    for i in (0, 1, 500, 999):
        h = 0x9E3779B1
        h = L.orc_xxh3_64(a[i:i + 1].ctypes.data, 4, h) & 0xFFFFFFFF
        h = L.orc_xxh3_64(b[i:i + 1].ctypes.data, 8, h) & 0xFFFFFFFF
        assert hv[i] == h and ch[i] == (h * 7) >> 32


def test_chunk_wire_format_bytes(oracle):
    # ChunkPB.data at encode level 0 (protobuf_serde.cpp:88-140, column_array_serde.cpp:228-238,768-772), written out by hand:
    # version 1, 3 rows; nullable int32 column = null column (uint8 x 3) then data column; int64 column
    a = np.array([7, -1, 300], dtype=np.int32)
    an = np.array([0, 1, 0], dtype=np.uint8)
    b = np.array([1, 2, -3], dtype=np.int64)
    got = oracle.chunk_serialize(Chunk([(5, a, an), (9, b, None)]))
    import struct
    want = struct.pack("<II", 1, 3) + struct.pack("<I", 3) + bytes([0, 1, 0]) + struct.pack("<I", 12) + struct.pack("<iii", 7, -1, 300) \
        + struct.pack("<I", 24) + struct.pack("<qqq", 1, 2, -3)
    assert got.tobytes() == want
    assert oracle.chunk_serialize(Chunk([(5, a, an), (9, b, None)]), 1, 2).tobytes() == \
        struct.pack("<II", 1, 1) + struct.pack("<I", 1) + bytes([1]) + struct.pack("<Ii", 4, -1) + struct.pack("<Iq", 8, 2)


def test_q95_plan_equals_join_free_evaluation(oracle):
    # TPC-DS Q95 shape (one-to-many self join, other conjunct, IN-subqueries, COUNT DISTINCT) through the oracle's operators
    # against the query evaluated without joins over the generator functions
    from starrocks_b200 import tpcds
    g = tpcds.Q95Gen(0.3)
    ws, wr = g.web_sales_of_orders(0, g.n_orders), g.web_returns_of_orders(0, g.n_orders)
    dims = {"date": Chunk([(tpcds.D_DATE_SK, g.date_keys(), None)]), "addr": Chunk([(tpcds.CA_ADDRESS_SK, g.address_keys(), None)]),
            "site": Chunk([(tpcds.WEB_SITE_SK, g.site_keys(), None)])}
    res, st = tpcds.q95_local_plan(tpcds.OracleEngine(oracle), tpcds.table_chunk(ws, tpcds.WS_COLS), Chunk([(tpcds.WS_ORDER, wr["wr_order_number"], None)]),
                                   dims, morsel_rows=50_000)
    assert res == g.expected(0, g.n_orders) and res[0] > 10
    assert st["self_join_rows"] > 10 * len(ws["ws_order_number"])          # the join really is one-to-many


def _for_cases(dt):
    rng = np.random.default_rng(17)
    info = np.iinfo(dt)
    yield "empty", np.zeros(0, dtype=dt)
    yield "one", np.array([2019], dtype=dt)
    yield "half_frame", np.arange(64, dtype=dt)                              # TestHalfFrame / TestOneFrame / TestTwoFrame ...
    yield "one_frame", np.arange(128, dtype=dt)
    yield "two_half_frames", np.arange(320, dtype=dt)
    yield "constant", np.full(300, 7, dtype=dt)
    yield "random_small_range", rng.integers(1000, 1000 + (1 << 22), 5000).astype(dt)      # SSB key columns: 22-bit deltas
    # delta overflow -> original values (storage format 2).  Single-frame pages only: the reference WRITER appends
    # n * bit_width BYTES for such a frame (frame_of_reference_coding.cpp:172-176, a bit count used as a byte count; the
    # tail is uninitialised memory) while its READER steps bit_width * 128 / 8 bytes (:266-272), so the reference cannot
    # read back its own page when another frame follows one of these.  Both restatements follow the reference as it is.
    yield "random_full_range", rng.integers(info.min, info.max, 100, dtype=dt)
    yield "negative", rng.integers(-500, 500, 777).astype(dt)
    yield "ascending_big_steps", np.cumsum(rng.integers(0, 1 << 20, 1000)).astype(dt)
    yield "ascending_then_not", np.concatenate([np.arange(128), rng.integers(0, 50, 128), np.arange(40)]).astype(dt)
    yield "extremes", np.array([info.min, info.max, 0, -1, 1, info.min, info.max] * 18, dtype=dt)
    yield "ascending_overflow", np.array([info.min, info.max] + [info.max] * 126, dtype=dt)


@pytest.mark.parametrize("dt", [np.int32, np.int64])
def test_for_page_codec_matches_the_reference_codec(oracle, dt):
    # the frame-of-reference pages stored in tests/golden (scripts/make_reference_vectors.py) against the restatement: the
    # encoded page bytes are identical and the restatement decodes them (cases follow
    # be/test/util/frame_of_reference_coding_test.cpp: half / one / two / two-and-a-half frames, int64, min value, zero
    # values).  Where `make -C oracle ref` built oracle/_ref/libfor_ref.so from the reference tree, the codec itself is
    # compared too: each side decodes the other's pages.
    g = np.load(GOLDEN)
    cases = [(name, g[f"for_{np.dtype(dt).name}_{name}_values"], g[f"for_{np.dtype(dt).name}_{name}_page"]) for name, _ in _for_cases(dt)]
    for name, v, page in cases:
        assert v.dtype == dt and oracle.for_encode(v).tobytes() == page.tobytes(), name
        assert (oracle.for_decode(page, dt) == v).all(), name
    ref = oracle.ref_for()
    if ref is None:
        return
    enc, dec = (ref.ref_for_encode_i32, ref.ref_for_decode_i32) if dt == np.int32 else (ref.ref_for_encode_i64, ref.ref_for_decode_i64)
    for name, v, mine in cases:
        buf = np.zeros(len(v) * (v.dtype.itemsize * 8 + 2) + 64, dtype=np.uint8)
        n = enc(v.ctypes.data if len(v) else None, len(v), buf.ctypes.data, len(buf))
        assert n > 0 and n == len(mine), name
        if name in ("random_full_range", "extremes", "ascending_overflow"):   # format 2: compare the defined bytes only
            used = v.dtype.itemsize * (1 + len(v))
            assert mine[-7:].tobytes() == bytes([2, 8 * v.dtype.itemsize, 128]) + len(v).to_bytes(4, "little"), name
            assert mine[:used].tobytes() == buf[:used].tobytes() and mine[-7:].tobytes() == buf[n - 7:n].tobytes(), name
        else:
            assert mine.tobytes() == buf[:n].tobytes(), name
        out = np.zeros(max(len(v), 1), dtype=dt)
        assert dec(mine.ctypes.data, len(mine), out.ctypes.data, len(out)) == len(v), name
        assert (out[:len(v)] == v).all(), name
        assert (oracle.for_decode(buf[:n], dt) == v).all(), name


@pytest.mark.parametrize("dt", [np.int32, np.int64])
def test_for_page_known_answers(oracle, dt):
    # frame_of_reference_coding_test.cpp TestZeroValue: an empty page is the 5-byte footer; the format itself
    # (frame_of_reference_coding.h:96-118): min, MSB-first deltas, (format, width) per frame, frame size 128, value count
    assert oracle.for_encode(np.zeros(0, dtype=dt)).tobytes() == bytes([128, 0, 0, 0, 0])
    page = oracle.for_encode(np.array([1, 2, 4, 8], dtype=dt) + 100)
    w = np.dtype(dt).itemsize
    # ascending -> deltas vs the predecessor 0,1,2,4 in 3 bits: 000 001 010 100 -> 0000 0101 0100 (0000)
    assert page.tobytes() == (101).to_bytes(w, "little") + bytes([0b00000101, 0b01000000]) + bytes([1, 3]) + bytes([128]) + (4).to_bytes(4, "little")
    assert (oracle.for_decode(page, dt) == np.array([101, 102, 104, 108], dtype=dt)).all()
    for name, v in _for_cases(dt):
        assert (oracle.for_decode(oracle.for_encode(v), dt) == v).all(), name
        assert (oracle.plain_decode(oracle.plain_encode(v), dt) == v).all(), name
    assert oracle.plain_encode(np.array([5, 6], dtype=np.int32)).tobytes() == bytes([2, 0, 0, 0, 5, 0, 0, 0, 6, 0, 0, 0])   # plain_page.h:82-86


def test_right_and_full_join_post_probe_known_answers(oracle):
    # build keys 1, 2, 2, 3, NULL (rows 1..5); probe keys 2, 4.  POST_PROBE (join_hash_map.hpp:420-457): build rows whose
    # build_match_index stayed 0, in build order; a NULL build key never matches
    bkey = np.array([1, 2, 2, 3, 0], dtype=np.int32)
    bnul = np.array([0, 0, 0, 0, 1], dtype=np.uint8)
    bpay = np.array([10, 20, 21, 30, 40], dtype=np.int32)
    build = Chunk([(10, bkey, bnul), (11, bpay, None)])
    probe = Chunk([(0, np.array([2, 4], dtype=np.int32), None), (1, np.array([100, 400], dtype=np.int64), None)])
    exp = {abi.JOIN_RIGHT_OUTER: ([(0, 3), (0, 2)], [10, 30, 40]), abi.JOIN_FULL_OUTER: ([(0, 3), (0, 2), (1, 0)], [10, 30, 40]),
           abi.JOIN_RIGHT_ANTI: ([], [10, 30, 40]), abi.JOIN_RIGHT_SEMI: ([], [20, 21])}
    for jt, (pairs, remain_pay) in exp.items():
        j = oracle.Join(abi.make_join_desc(jt, [10], [0], [abi.TYPE_INT], build_out=[11], probe_out=[1]))
        j.append_build(build)
        j.build()
        pi, bi = j.probe_all(probe)
        assert list(zip(pi.tolist(), bi.tolist())) == pairs, jt          # chain order: descending build index, like INNER
        rem = j.probe_remain([abi.TYPE_BIGINT])
        assert rem[-1][1].tolist() == remain_pay, jt
        if jt in (abi.JOIN_RIGHT_OUTER, abi.JOIN_FULL_OUTER):
            assert rem[0][0] == 1 and rem[0][2].tolist() == [1] * len(remain_pay)      # probe column: all NULL
        else:
            assert len(rem) == 1


def test_other_join_conjunct_known_answers(oracle):
    # build (key, b): (1, 5) (1, 9) (2, 7) (3, 1); probe (key, a): (1, 6) (2, 8) (4, 0) (3, 0).  Conjunct a < b.
    # candidates by key: p0-{b2 (9), b1 (5)}, p1-{b3 (7)}, p3-{b4 (1)}; passing: p0-b2 (6 < 9) and p3-b4 (0 < 1).
    build = Chunk([(10, np.array([1, 1, 2, 3], dtype=np.int32), None), (11, np.array([5, 9, 7, 1], dtype=np.int32), None)])
    probe = Chunk([(0, np.array([1, 2, 4, 3], dtype=np.int32), None), (1, np.array([6, 8, 0, 0], dtype=np.int32), None)])
    conj = [("col", 1), ("col", 11), "<"]
    exp = {abi.JOIN_INNER: [(0, 2), (3, 4)], abi.JOIN_LEFT_OUTER: [(0, 2), (1, 0), (2, 0), (3, 4)], abi.JOIN_LEFT_SEMI: [(0, 0), (3, 0)],
           abi.JOIN_LEFT_ANTI: [(1, 0), (2, 0)], abi.JOIN_RIGHT_OUTER: [(0, 2), (3, 4)], abi.JOIN_FULL_OUTER: [(0, 2), (1, 0), (2, 0), (3, 4)],
           abi.JOIN_RIGHT_ANTI: [], abi.JOIN_RIGHT_SEMI: []}
    remain = {abi.JOIN_RIGHT_OUTER: [5, 7], abi.JOIN_FULL_OUTER: [5, 7], abi.JOIN_RIGHT_ANTI: [5, 7], abi.JOIN_RIGHT_SEMI: [9, 1]}
    for jt, pairs in exp.items():
        j = oracle.Join(abi.make_join_desc(jt, [10], [0], [abi.TYPE_INT], build_out=[11], probe_out=[1], other_conjunct=conj))
        j.append_build(build)
        j.build()
        pi, bi = j.probe_all(probe)
        assert list(zip(pi.tolist(), bi.tolist())) == pairs, jt
        if jt in remain:
            assert j.probe_remain([abi.TYPE_INT])[-1][1].tolist() == remain[jt], jt


def test_exchange_and_join_hashes_against_the_reference_functions(oracle):
    # HashUtil::fnv_hash / zlib_crc_hash (hash_util.hpp:34-45,127-134) and crc_hash_32 (hash.h:96-130) against the
    # restatements, on random byte strings of every length 0..40 and a few long ones, three seeds each.  The known answers
    # (tests/golden, written by scripts/make_reference_vectors.py) come from FNV-1a, zlib's crc32 and CRC-32C; where
    # `make -C oracle ref` built oracle/_ref/libhash_ref.so from the reference tree, the reference functions are held to them too.
    g = np.load(GOLDEN)
    o = oracle.lib()
    ref = oracle.ref_hash()
    impls = [("fnv_hash", o.orc_fnv_hash), ("zlib_crc_hash", o.orc_zlib_crc32), ("crc_hash_32", o.orc_crc_hash_32)]
    if ref is not None:
        impls += [("fnv_hash", ref.ref_fnv_hash), ("zlib_crc_hash", ref.ref_zlib_crc_hash), ("crc_hash_32", ref.ref_crc_hash_32)]
    data = g["hash_bytes"]
    for i, (off, n, seed) in enumerate(zip(g["hash_buf_offset"].tolist(), g["hash_len"].tolist(), g["hash_seed"].tolist())):
        b = np.ascontiguousarray(data[off:off + max(n, 1)])
        for key, fn in impls:
            assert fn(b.ctypes.data, n, seed) == int(g[key][i]), (fn.__name__, n, seed)


@pytest.mark.parametrize("with_conjunct", [False, True])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_join_types_against_a_row_at_a_time_definition(oracle, seed, with_conjunct):
    # every join type (probe phase + POST_PROBE rows) against the textbook definition evaluated row by row in Python: the equi
    # key with SQL NULL semantics (NULL never equals), the other-join conjunct a < b with NULL = false, duplicates on both sides
    rng = np.random.default_rng(seed)
    nb, npr = 60, 90
    bk, pk = rng.integers(0, 12, nb).astype(np.int32), rng.integers(-1, 14, npr).astype(np.int32)
    bkn, pkn = (rng.random(nb) < 0.1).astype(np.uint8), (rng.random(npr) < 0.1).astype(np.uint8)
    bv, pv = rng.integers(0, 10, nb).astype(np.int32), rng.integers(0, 10, npr).astype(np.int32)
    bvn, pvn = (rng.random(nb) < 0.15).astype(np.uint8), (rng.random(npr) < 0.15).astype(np.uint8)
    build = Chunk([(10, bk, bkn), (11, bv, bvn)])
    probe = Chunk([(0, pk, pkn), (1, pv, pvn)])

    def match(i, b):      # probe row i joins build row b
        if pkn[i] or bkn[b] or pk[i] != bk[b]:
            return False
        if with_conjunct and (pvn[i] or bvn[b] or not pv[i] < bv[b]):
            return False
        return True

    P = lambda i: (None if pkn[i] else int(pk[i]), None if pvn[i] else int(pv[i]))
    B = lambda b: (None if bkn[b] else int(bk[b]), None if bvn[b] else int(bv[b]))
    NP, NB = (None, None), (None, None)
    pairs = [(i, b) for i in range(npr) for b in range(nb) if match(i, b)]
    p_any = {i for i, _ in pairs}
    b_any = {b for _, b in pairs}
    want = {
        abi.JOIN_INNER: [P(i) + B(b) for i, b in pairs],
        abi.JOIN_LEFT_OUTER: [P(i) + B(b) for i, b in pairs] + [P(i) + NB for i in range(npr) if i not in p_any],
        abi.JOIN_LEFT_SEMI: [P(i) for i in range(npr) if i in p_any],
        abi.JOIN_LEFT_ANTI: [P(i) for i in range(npr) if i not in p_any],
        abi.JOIN_RIGHT_OUTER: [P(i) + B(b) for i, b in pairs] + [NP + B(b) for b in range(nb) if b not in b_any],
        abi.JOIN_FULL_OUTER: [P(i) + B(b) for i, b in pairs] + [P(i) + NB for i in range(npr) if i not in p_any] + [NP + B(b) for b in range(nb) if b not in b_any],
        abi.JOIN_RIGHT_SEMI: [B(b) for b in range(nb) if b in b_any],
        abi.JOIN_RIGHT_ANTI: [B(b) for b in range(nb) if b not in b_any],
    }
    key = lambda r: tuple((0, 0) if v is None else (1, v) for v in r)
    for jt, exp in want.items():
        d = abi.make_join_desc(jt, [10], [0], [abi.TYPE_INT], build_out=[10, 11], probe_out=[0, 1],
                               other_conjunct=[("col", 1), ("col", 11), "<"] if with_conjunct else None)
        j = oracle.Join(d)
        j.append_build(build)
        j.build()
        got = []
        for lo, hi in ((0, 40), (40, npr)):         # two probe calls: marks accumulate across them
            ch = Chunk([(s, a[lo:hi].copy(), nl[lo:hi].copy()) for s, a, nl in probe.columns()])
            pi, bi = j.probe_all(ch)
            cols = j.output(ch, pi, bi)
            vals = [[None if nl[q] else int(a[q]) for q in range(len(pi))] for _, a, nl in cols]
            got += list(zip(*vals)) if vals and len(pi) else []
        if jt in (abi.JOIN_RIGHT_OUTER, abi.JOIN_FULL_OUTER, abi.JOIN_RIGHT_SEMI, abi.JOIN_RIGHT_ANTI):
            rem = j.probe_remain([abi.TYPE_INT, abi.TYPE_INT])
            n = len(rem[0][1])
            vals = [[None if nl[q] else int(a[q]) for q in range(n)] for _, a, nl in rem]
            got += list(zip(*vals)) if n else []
        if jt in (abi.JOIN_RIGHT_SEMI, abi.JOIN_RIGHT_ANTI):
            got = [r[-2:] for r in got]
        assert sorted(got, key=key) == sorted(exp, key=key), (jt, with_conjunct)

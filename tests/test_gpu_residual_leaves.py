"""Residual leaves (-m gpu): when the aggregation runs in pb_agg_rows_kernel, a dictionary leaf of a flat AND that would be
tested on the filter kernel's candidates, and whose column is a field of the row group, is tested by the rows kernel on the
row it loads anyway (DevRowLeaf).  The filter kernel then hands its survivors over as candidates, and numDocsScanned is
counted by the rows kernel.  Results and statistics must equal the oracle's, and Result.residual_leaves tells which path
ran."""
import numpy as np
import pytest

from oracle import oracle
from pinot_b200 import native
from pinot_b200.query import parse_sql
from pinot_b200.segment_writer import DataType, build_dict_column, make_segment
from tests.parity import assert_rows_equal, check_query, combined_rows, oracle_rows

pytestmark = pytest.mark.gpu
ALL_FLAGS = (0, native.PB_Q_GENERIC_KERNEL, native.PB_Q_NO_TMA)
N = 300_017


@pytest.fixture(scope="module")
def table():
    native.init()
    rng = np.random.default_rng(11)
    # a: 1000 values, skewed: 70 % of the docs carry dictId 3 (the statistics say 0.1 %)
    a_ids = rng.integers(0, 1000, N, dtype=np.uint32)
    a_ids[rng.random(N) < 0.7] = 3
    a_ids[:1000] = np.arange(1000, dtype=np.uint32)
    a_vals = np.arange(1000, dtype=np.int32) * 7 + 1
    b_ids = rng.integers(0, 5000, N, dtype=np.uint32); b_ids[:5000] = np.arange(5000, dtype=np.uint32)
    b = build_dict_column("b", DataType.INT, np.arange(5000, dtype=np.int32) * 3, b_ids)
    c_ids = rng.integers(0, 20000, N, dtype=np.uint32); c_ids[:20000] = np.arange(20000, dtype=np.uint32)   # > 8192 entries
    c = build_dict_column("c", DataType.LONG, np.arange(20000, dtype=np.int64) * 1_000_003, c_ids)
    d = build_dict_column("d", DataType.INT, np.arange(6, dtype=np.int32) + 10, rng.integers(0, 6, N, dtype=np.uint32))
    m = build_dict_column("m", DataType.INT, np.arange(50_000, dtype=np.int32) * 2,
                          np.concatenate([np.arange(50_000, dtype=np.uint32), rng.integers(0, 50_000, N - 50_000, dtype=np.uint32)]))
    segs = []
    for i, ids in enumerate((a_ids, a_ids[::-1].copy())):
        # e: 0 for the docs whose a has dictId < 500, else 1 -- "a among the first 500 values AND e = 1" matches nothing
        e = build_dict_column("e", DataType.INT, np.array([0, 1], dtype=np.int32), (ids >= 500).astype(np.uint32))
        segs.append(make_segment(f"resid{i}", [build_dict_column("a", DataType.INT, a_vals, ids), b, c, d, e, m]))
    staged = [native.StagedSegment(s) for s in segs]
    group = native.SegmentGroup(staged)
    yield segs, group
    group.release()
    for s in staged:
        s.release()


def _scan_leaves(group, q):
    return sum(1 for ln in native.dump_lowered(group, q) if ln.startswith("SCAN_"))


def _check(segs, group, sql, residual_per_segment, flags_list=ALL_FLAGS):
    check_query(segs, sql, group=group, flags_list=flags_list)
    q = parse_sql(sql)
    n_scan = _scan_leaves(group, q)
    for flags in flags_list:
        for combine in (0, native.PB_Q_COMBINE):
            res = native.execute(group, q, flags | combine)
            assert res.residual_leaves == residual_per_segment * len(segs), (sql, flags, combine, res.residual_leaves)
            # the streamed and the residual leaves both count as reading every doc, as before
            assert sum(t.stats["num_entries_scanned_in_filter"] for t in res.tables) == n_scan * sum(s.num_docs for s in segs)
            res.free()


def test_dictionary_range(table):
    segs, group = table
    _check(segs, group, "SELECT d, COUNT(*), SUM(m), MIN(m), MAX(m), AVG(m) FROM t WHERE a IN (8, 15, 29, 701) AND b < 9000 GROUP BY d", 1)


def test_in_small_and_large_sets_and_not_in(table):
    segs, group = table
    c_in = ", ".join(str(v * 1_000_003) for v in range(0, 20000, 2))          # 10 000 entries of a 20 000-entry dictionary
    _check(segs, group, "SELECT d, COUNT(*), SUM(m) FROM t WHERE a IN (8, 15, 29, 701) AND d IN (10, 12) GROUP BY d", 1)
    _check(segs, group, f"SELECT d, COUNT(*), MAX(m) FROM t WHERE a IN (8, 15, 29, 701) AND c IN ({c_in}) GROUP BY d", 1)
    _check(segs, group, "SELECT d, COUNT(*), SUM(m) FROM t WHERE a IN (8, 15, 29, 701) AND b NOT IN (3, 6, 9, 12, 300) GROUP BY d", 1)


def test_two_residual_leaves(table):
    segs, group = table
    _check(segs, group, "SELECT d, COUNT(*), SUM(m), MIN(m) FROM t WHERE a IN (8, 15, 29, 701) AND b BETWEEN 300 AND 12000 AND d IN (11, 13, 14) GROUP BY d", 2)


def test_skewed_column_many_candidates(table):
    # a = 22 is dictId 3: the statistics expect 0.1 % of the docs, 70 % arrive as candidates
    segs, group = table
    _check(segs, group, "SELECT d, COUNT(*), SUM(m), MAX(m) FROM t WHERE a = 22 AND b < 9000 GROUP BY d", 1)


def test_every_candidate_fails(table):
    segs, group = table
    in_list = ", ".join(str(v * 7 + 1) for v in range(0, 500, 50))
    sql = f"SELECT d, COUNT(*), SUM(m) FROM t WHERE a IN ({in_list}) AND e = 1 GROUP BY d"
    _check(segs, group, sql, 1)
    res = native.execute(group, parse_sql(sql), native.PB_Q_COMBINE)
    assert res.tables[0].num_groups == 0 and res.tables[0].stats["num_docs_scanned"] == 0
    res.free()


def test_num_groups_limit_keeps_the_first_groups_in_doc_order(table):
    segs, group = table
    for limit in (1, 3, 5):
        q = parse_sql(f"SET numGroupsLimit = {limit}; SELECT d, COUNT(*), SUM(m), MIN(m) FROM t WHERE a IN (8, 15, 29, 701) AND b < 9000 GROUP BY d")
        for flags in (0, native.PB_Q_GENERIC_KERNEL):
            res = native.execute(group, q, flags)
            assert res.residual_leaves == len(segs)
            for i, (t, s) in enumerate(zip(res.tables, segs)):
                o = oracle.execute(s, q)
                assert_rows_equal(t.rows(), oracle_rows(o), q, exact_float=True, what=f"limit {limit} segment {i}")
                for key in ("num_groups_limit_reached", "num_docs_scanned", "num_entries_scanned_post_filter"):
                    assert t.stats[key] == o.stats[key], (limit, key, t.stats, o.stats)
            res.free()


def test_plan_cache_replays(table):
    # build, eager replay, graph capture, then graph launches (every 8th replay is eager again)
    segs, group = table
    q = parse_sql("SELECT d, COUNT(*), SUM(m), MAX(m) FROM t WHERE a IN (8, 15, 29, 701) AND b < 9000 AND d <> 12 GROUP BY d")
    orc = [oracle.execute(s, q) for s in segs]
    exp = combined_rows(oracle.combine(orc), q)
    for flags in (native.PB_Q_COMBINE, 0):
        for run in range(10):
            r = native.execute(group, q, flags)
            assert r.residual_leaves == 2 * len(segs)
            if flags:
                assert_rows_equal(r.tables[0].rows(), exp, q, exact_float=True, what=f"combined run {run}")
                assert r.tables[0].stats["num_docs_scanned"] == sum(o.stats["num_docs_scanned"] for o in orc)
            else:
                for i, (t, o) in enumerate(zip(r.tables, orc)):
                    assert_rows_equal(t.rows(), oracle_rows(o), q, exact_float=True, what=f"run {run} segment {i}")
                    for key in ("num_docs_scanned", "num_entries_scanned_post_filter"):
                        assert t.stats[key] == o.stats[key]
            r.free()


def test_other_paths_keep_their_candidates(table):
    # no rows kernel (keyless, DISTINCTCOUNT): the candidate leaves stay in the filter kernel
    segs, group = table
    for sql in ("SELECT COUNT(*), SUM(m) FROM t WHERE a IN (8, 15, 29, 701) AND b < 9000",
                "SELECT d, DISTINCTCOUNT(m) FROM t WHERE a IN (8, 15, 29, 701) AND b < 9000 GROUP BY d"):
        check_query(segs, sql, group=group)
        res = native.execute(group, parse_sql(sql), native.PB_Q_COMBINE)
        assert res.residual_leaves == 0
        res.free()

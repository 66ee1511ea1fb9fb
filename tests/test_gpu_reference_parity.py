"""GPU operators against the reference's answers (unmodified DuckDB, recorded in tests/golden/reference_answers.json)
at SF1-like sizes, on rows both sides generate from the same formulas (bench_data.py): TPC-H Q1 / Q14 shapes at SF1
(6 M rows) and the group-by at the three cardinalities of the BASELINE configs - 35 groups (SSB Q4.1), 11 620 groups
(Q3 at SF1) and 3.5 M groups (Q3 at SF300).  Integer results bit-exact, AVG within 1e-9 relative (BASELINE.json
north_star)."""
import numpy as np
import pytest
import torch

import bench_data as BD
from conftest import digest, reference_answers
from duckdb_b200 import capi
from duckdb_b200 import operators as ops

pytestmark = pytest.mark.gpu

SF1_LINEITEM = 6_001_215
Q14_PART_ROWS = 200_000
Q1_SQL = ("SELECT rf, ls, sum(qty), sum(price), sum(disc_price), sum(charge), avg(qty), avg(price), avg(disc), "
          "count(*) FROM q1in GROUP BY rf, ls")
Q14_SQL = ("SELECT count(*), sum(price), sum(disc), sum(promo), sum(li.partkey * promo) FROM li JOIN part "
           "ON li.partkey = part.partkey")
GROUPBY_CASES = [(35, 3_000_000, "ssb"), (11_620, 3_000_000, "q3"), (3_500_000, 9_000_000, "q3"),
                 (3_500_000, 9_000_000, "q3wide")]
GROUPBY_SQL = {"ssb": "SELECT year, nation, sum(profit), count(*) FROM t GROUP BY year, nation",
               "q3": "SELECT okey, odate, prio, sum(revenue), count(*) FROM t GROUP BY okey, odate, prio"}


def groupby_key(groups, n, keytypes):
    return f"{keytypes}_{groups}_{n}"


def groupby_digests(cols, nk):
    """canonical form of a group-by result: rows sorted by the keys, every column as int64 -> {column: digest}"""
    cols = [np.array([int(v) for v in c], dtype=np.int64) if c.dtype == object else c.astype(np.int64) for c in cols]
    order = np.lexsort(cols[:nk][::-1])
    return {"groups": len(order), "columns": [digest(c[order]) for c in cols]}


def upload(ctx, cols):
    arrs = [c.numpy() for c in cols]
    return ops.Batch.upload(ctx, [ops.Vector.flat(a) for a in arrs], len(arrs[0]))


def test_q1_sf1_vs_reference(ctx):
    n = SF1_LINEITEM
    d = BD.Gen(torch, "cpu").q1(n)
    desc = [(capi.AGG_SUM, capi.INT64, 0), (capi.AGG_SUM, capi.INT64, 1), (capi.AGG_SUM, capi.INT64, 2),
            (capi.AGG_SUM, capi.INT64, 3), (capi.AGG_AVG, capi.INT64, 0), (capi.AGG_AVG, capi.INT64, 1),
            (capi.AGG_AVG, capi.INT64, 4), (capi.AGG_COUNT_STAR, capi.INT64, -1)]
    a = ops.HashAggregate(ctx, [capi.UINT8, capi.UINT8], desc)
    a.sink(upload(ctx, [d[k] for k in ("rf", "ls", "qty", "price", "disc_price", "charge", "disc")]), [0, 1], [2, 3, 4, 5, 6])
    res = a.finalize().download_all()
    rows = [tuple(r) for r in reference_answers("gpu_q1_sf1")]
    got = {(int(res[0][0][g]), int(res[1][0][g])): [res[2 + i][0][g] for i in range(8)] for g in range(len(res[0][0]))}
    assert len(got) == len(rows) == 4
    for r in rows:
        g = got[(r[0], r[1])]
        assert [int(x) for x in g[:4]] == [int(x) for x in r[2:6]] and int(g[7]) == int(r[9])
        for x, y in zip(g[4:7], r[6:9]):
            assert float(x) == pytest.approx(float(y), rel=1e-9)


@pytest.mark.parametrize("no_dense", [False, True])
def test_q14_sf1_vs_reference(ctx, monkeypatch, no_dense):
    """600 K part rows x 6 M lineitem rows; no_dense forces the open-addressing table (LEAN probe kernel on it)."""
    if no_dense:
        monkeypatch.setenv("B200_JOIN_NO_DENSE", "1")
    n, nb = SF1_LINEITEM, Q14_PART_ROWS
    g = BD.Gen(torch, "cpu")
    part, probe = g.part(nb, 1), g.probe(n, nb)
    j = ops.HashJoin(ctx, capi.JOIN_INNER, [capi.INT64], [capi.UINT8])
    j.sink(upload(ctx, [part["partkey"], part["promo"]]), [0], [1])
    j.finalize()
    out, cnt = j.execute(upload(ctx, [probe["partkey"], probe["price"], probe["disc"]]), [0], [0, 1, 2])
    res = out.download_all()
    r = reference_answers("gpu_q14_sf1")
    k, price, disc, promo = (res[i][0] for i in range(4))
    assert cnt == int(r[0]) == n
    assert int(price.astype(object).sum()) == int(r[1]) and int(disc.sum()) == int(r[2]) and int(promo.sum()) == int(r[3])
    assert int((k.astype(object) * promo.astype(object)).sum()) == int(r[4])


@pytest.mark.parametrize("groups,n,keytypes", GROUPBY_CASES)
def test_groupby_cardinalities_vs_reference(ctx, groups, n, keytypes):
    """35 groups -> thread-private shared-memory path, 11 620 / 3.5 M groups -> the L2-first high-cardinality table
    (q3wide: BIGINT + INTEGER + INTEGER keys = three key words)."""
    g = BD.Gen(torch, "cpu")
    if keytypes == "ssb":
        d = g.ssb(n)
        cols, types, nk = [d["year"], d["nation"], d["profit"]], [capi.INT32, capi.UINT8, capi.INT64], 2
    else:
        d = g.q3(n, groups)
        cols = [d["okey"], d["odate"], d["prio"], d["revenue"]]
        types, nk = [capi.INT64, capi.UINT16, capi.UINT8, capi.INT64], 3
        if keytypes == "q3wide":
            cols = [d["okey"], d["odate"].to(torch.int32), d["prio"].to(torch.int32), d["revenue"]]
            types = [capi.INT64, capi.INT32, capi.INT32, capi.INT64]
    a = ops.HashAggregate(ctx, types[:nk], [(capi.AGG_SUM, capi.INT64, 0), (capi.AGG_COUNT_STAR, capi.INT64, -1)])
    half = n // 2 // 1024 * 1024
    for lo, hi in ((0, half), (half, n)):   # two batches: the second one meets an existing table
        a.sink(upload(ctx, [c[lo:hi] for c in cols]), list(range(nk)), [nk])
    res = a.finalize().download_all()
    want = reference_answers("gpu_groupby")[groupby_key(groups, n, keytypes)]
    got = groupby_digests([res[j][0] for j in range(nk + 2)], nk)
    assert got["groups"] == want["groups"]
    assert got["columns"] == want["columns"]

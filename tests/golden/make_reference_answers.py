#!/usr/bin/env python3
"""Record what the UNMODIFIED reference answers for the tests that compare with it, into reference_answers.json.

    python oracle/build_ref.py                      # oracle/_ref/libduckdb_ref.so from the DuckDB sources
    DUCKDB_REF=<duckdb source tree> python tests/golden/make_reference_answers.py

The tests build the same seeded inputs (the table functions and SQL below are theirs) and compare their results
with these answers, so they need neither the reference library nor its sources.  Small results are stored as rows;
large ones as conftest.digest() of the canonical form the test computes.
"""
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]
import bench_data as BD  # noqa: E402
import test_bench_data as TBD  # noqa: E402
import test_gpu_parity as TGP  # noqa: E402
import test_gpu_reference_parity as TGR  # noqa: E402
import test_oracle as TO  # noqa: E402
from conftest import digest  # noqa: E402
from oracle import duckdb_ref as R  # noqa: E402

REF = os.environ.get("DUCKDB_REF", "/root/reference")


def header_enum(path, enum_name):
    """{NAME: value} of `enum class <enum_name>` in a reference header (C rules: previous + 1 when not explicit)."""
    text = open(os.path.join(REF, path)).read()
    m = re.search(r"enum class " + enum_name + r"\b[^{]*\{(.*?)\};", text, re.S)
    assert m, f"{enum_name} not found in {path}"
    body = re.sub(r"//[^\n]*", "", m.group(1))
    values, nxt = {}, 0
    for item in body.split(","):
        m = re.match(r"\s*([A-Z_0-9]+)\s*(?:=\s*(\d+))?\s*$", item)
        if not m:
            continue
        nxt = int(m.group(2)) if m.group(2) is not None else nxt
        values[m.group(1)] = nxt
        nxt += 1
    return values


def enums():
    inc = "src/include/duckdb/common/"
    return {"PhysicalType": header_enum(inc + "types.hpp", "PhysicalType"),
            "ExpressionType": header_enum(inc + "enums/expression_type.hpp", "ExpressionType"),
            "JoinType": header_enum(inc + "enums/join_type.hpp", "JoinType"),
            "VectorType": header_enum(inc + "enums/vector_type.hpp", "VectorType")}


def port_groupby(con):
    con.load_table("pg", TO.pg_table())
    h = con.execute("SELECT hash(k1, k2) FROM pg")[0].values
    con.execute("SET perfect_ht_threshold=0")
    rows = con.fetchall(TO.PG_GROUPBY_SQL)
    con.execute("RESET perfect_ht_threshold")
    return {"hash": digest(h), "rows": rows}


def port_joins(con):
    jb, jp = TO.join_tables()
    con.load_table("jb", jb)
    con.load_table("jp", jp)
    out = {}
    for i, keys_sql in enumerate(TO.JOIN_KEYS_SQL):
        out[f"inner{i}"] = TO.join_digest(con.fetchall(f"SELECT jp.id, jb.id FROM jp JOIN jb ON {keys_sql}"))
        left = con.fetchall(f"SELECT jp.id, jb.id FROM jp LEFT JOIN jb ON {keys_sql}")
        out[f"left{i}"] = TO.join_digest([(a, -1 if b is None else b) for a, b in left])
        out[f"semi{i}"] = TO.join_digest([r[0] for r in con.fetchall(f"SELECT jp.id FROM jp SEMI JOIN jb ON {keys_sql}")])
        out[f"anti{i}"] = TO.join_digest([r[0] for r in con.fetchall(f"SELECT jp.id FROM jp ANTI JOIN jb ON {keys_sql}")])
    mark = con.fetchall("SELECT id, k IN (SELECT k FROM jb) FROM jp ORDER BY id")
    out["mark"] = digest(np.array([-1 if m is None else int(bool(m)) for _, m in mark], dtype=np.int64))
    fb, fp = TO.FLOAT_JOIN_KEYS
    con.load_table("fjb", {"k": fb, "id": np.arange(len(fb), dtype=np.int32)})
    con.load_table("fjp", {"k": fp, "id": np.arange(len(fp), dtype=np.int32)})
    out["float_inner"] = sorted(con.fetchall("SELECT fjp.id, fjb.id FROM fjp JOIN fjb ON fjp.k = fjb.k"))
    return out


def port_filters(con):
    con.load_table("fl", TO.fl_table())
    return {sql: TO.join_digest([r[0] for r in con.fetchall(f"SELECT id FROM fl WHERE {sql}")]) for sql in TO.FL_CASES}


def bench_data(con):
    def table(sql):
        con.execute("DROP TABLE IF EXISTS t")
        con.execute(sql)
        return {c.name: c.values for c in con.execute("SELECT * FROM t")}

    out = {}
    for offset in (0, 591_855_000 * 3 + 12345):
        cols = table(BD.q1_table_sql("t", TBD.Q1_ROWS, offset))
        out[f"q1_{offset}"] = TBD.column_digests({k: cols[k] for k in TBD.Q1_COLUMNS})
        out[f"q1_{offset}"].update(rf_values=sorted(int(v) for v in np.unique(cols["rf"])),
                                   ls_values=sorted(int(v) for v in np.unique(cols["ls"])))
    for name, (sql, _) in TBD.OTHER_TABLES.items():
        out[name] = TBD.column_digests(table(sql))
    return out


def gpu_groupby_join(con):
    lr, ld = TGP.lr_tables()
    con.load_table("lr", lr)
    con.load_table("ld", ld)
    con.execute("SET perfect_ht_threshold=0")
    cols = con.execute(TGP.LR_GROUPBY_SQL)
    con.execute("RESET perfect_ht_threshold")
    ints = [np.array([int(v) for v in cols[i].values], dtype=np.int64) for i in (0, 1, 2, 4)]
    out = {"groups": len(ints[0]), "k": digest(ints[0]), "sum": digest(ints[1]), "min": digest(ints[2]),
           "count": digest(ints[3]), "avg_sample": [float(v) for v in cols[3].values[::TGP.LR_AVG_SAMPLE]]}
    out["join"] = [int(v) for v in con.fetchall(TGP.LR_JOIN_SQL)[0]]
    return out


def gpu_sf1(con):
    n, nb = TGR.SF1_LINEITEM, TGR.Q14_PART_ROWS
    con.execute(BD.q1_table_sql("q1in", n))
    q1 = con.fetchall(TGR.Q1_SQL)
    con.execute("DROP TABLE q1in")
    con.execute(BD.probe_table_sql("li", n, nb))
    con.execute(BD.part_table_sql("part", nb))
    q14 = list(con.fetchall(TGR.Q14_SQL)[0])
    con.execute("DROP TABLE li")
    con.execute("DROP TABLE part")
    groupby = {}
    for groups, n, keytypes in TGR.GROUPBY_CASES:
        kind = "ssb" if keytypes == "ssb" else "q3"   # q3wide: the same rows, wider key types on the GPU only
        con.execute("DROP TABLE IF EXISTS t")
        con.execute(BD.ssb_table_sql("t", n) if kind == "ssb" else BD.q3_table_sql("t", n, groups))
        cols = con.execute(TGR.GROUPBY_SQL[kind])
        groupby[TGR.groupby_key(groups, n, keytypes)] = TGR.groupby_digests([c.values for c in cols], len(cols) - 2)
    return q1, q14, groupby


def main():
    con = R.Connection(threads=os.cpu_count())
    q1, q14, groupby = gpu_sf1(con)
    out = {"enums": enums(), "port_groupby": port_groupby(con), "port_joins": port_joins(con),
           "port_filters": port_filters(con), "bench_data": bench_data(con), "gpu_groupby_join": gpu_groupby_join(con),
           "gpu_q1_sf1": q1, "gpu_q14_sf1": q14, "gpu_groupby": groupby}
    con.close()
    path = os.path.join(HERE, "reference_answers.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()

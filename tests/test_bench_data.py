"""bench.py's synthetic columns are defined as DuckDB SQL and restated with torch ops (bench_data.py): both arms of the
benchmark must see the same rows.  Pinned here against the reference's tables built from that SQL (digests of every
column in tests/golden/reference_answers.json)."""
import numpy as np
import pytest
import torch

import bench_data as BD
from conftest import digest, reference_answers

Q1_ROWS = 50_000
Q1_COLUMNS = ("rf", "ls", "qty", "price", "disc_price", "charge", "disc")
N, NB, GROUPS = 40_000, 1000, 5000
OTHER_TABLES = {   # name -> (the reference's table, the same rows from bench_data's torch generator)
    "ssb": (BD.ssb_table_sql("t", N, 77), lambda g: g.ssb(N, 77)),
    "q3": (BD.q3_table_sql("t", N, GROUPS, 5), lambda g: g.q3(N, GROUPS, 5)),
    "probe": (BD.probe_table_sql("t", N, NB, 3), lambda g: g.probe(N, NB, 3)),
    "part": (BD.part_table_sql("t", NB, 1001), lambda g: g.part(NB, 1001)),
    "scan": (BD.scan_table_sql("t", N, 9), lambda g: g.scan(N, 9)),
}


def column_digests(cols):
    return {k: digest(np.asarray(v).astype(np.int64)) for k, v in cols.items()}


@pytest.mark.parametrize("offset", [0, 591_855_000 * 3 + 12345])
def test_q1_columns_match_reference(offset):
    want = reference_answers("bench_data")[f"q1_{offset}"]
    got = BD.Gen(torch, "cpu", chunk=7777).q1(Q1_ROWS, offset)
    got = column_digests({k: got[k].numpy() for k in Q1_COLUMNS})
    for k in Q1_COLUMNS:
        assert got[k] == want[k], k
    assert set(want["rf_values"]) == {65, 78, 82} and set(want["ls_values"]) == {70, 79}


def test_other_tables_match_reference():
    want = reference_answers("bench_data")
    g = BD.Gen(torch, "cpu", chunk=9999)
    for name, (_, gen) in OTHER_TABLES.items():
        got = column_digests({k: v.numpy() for k, v in gen(g).items()})
        assert got == want[name], name


def test_effective_cores():
    cores, info = BD.effective_cores()
    assert 1 <= cores <= info["sched_affinity"]

"""The CPU oracle (oracle/port.py) pinned against the reference's own known-answer vectors, the golden
fixtures generated from the unmodified reference, and the reference's recorded answers on seeded random tables."""
import numpy as np
import pytest

from conftest import digest, golden, reference_answers
from oracle import port as P


def test_murmur_kat_from_reference_tests():
    # test/sql/function/generic/hash_func.test:160-171 (uint8 / enum values 0,1,2,3) and :22 (NULL)
    h = P.hash_values(np.array([0, 1, 2, 3], dtype=np.uint8))
    assert [int(x) for x in h] == [0, 4717996019076358352, 2060787363917578834, 8131803788478518982]
    assert int(P.NULL_HASH) == 13787848793156543929
    hv = P.hash_columns([(np.array([5], dtype=np.int32), np.array([False]))])
    assert int(hv[0]) == 13787848793156543929


@pytest.mark.parametrize("name", ["i8", "i16", "i32", "i64", "u8", "u16", "u32", "u64", "f32", "f64"])
def test_hash_golden(name):
    g = golden("hash_kat.npz")
    h = P.hash_columns([(g[f"{name}_v"], g[f"{name}_valid"])])
    np.testing.assert_array_equal(h, g[f"{name}_h"])


def test_hash_bool_and_multi_golden():
    g = golden("hash_kat.npz")
    np.testing.assert_array_equal(P.hash_columns([(g["bool_v"], None)]), g["bool_h"])
    h = P.hash_columns([(g["multi_a"], g["multi_a_valid"]), (g["multi_b"], g["multi_b_valid"]), (g["multi_c"], None)])
    np.testing.assert_array_equal(h, g["multi_h"])


FILTERS = {
    "lt_const": ("lt", ("col", 0), ("const", 7, np.int32)),
    "eq_cols": ("eq", ("col", 0), ("col", 1)),
    "ne_cols": ("ne", ("col", 0), ("col", 1)),
    "ge_cols": ("ge", ("col", 0), ("col", 1)),
    "and2": ("and", ("lt", ("col", 0), ("const", 10, np.int32)), ("gt", ("col", 1), ("const", -10, np.int32))),
    "or2": ("or", ("lt", ("col", 0), ("const", -20, np.int32)), ("gt", ("col", 1), ("const", 20, np.int32))),
    "and_or": ("or", ("and", ("lt", ("col", 0), ("const", 0, np.int32)), ("gt", ("col", 1), ("const", 0, np.int32))),
               ("eq", ("col", 0), ("col", 1))),
    "isnull": ("isnull", ("col", 0)),
    "isnotnull_and": ("and", ("isnotnull", ("col", 0)), ("lt", ("col", 1), ("const", 3, np.int32))),
    "distinct": ("distinct", ("col", 0), ("col", 1)),
    "notdistinct": ("notdistinct", ("col", 0), ("col", 1)),
    "dbl_gt": ("gt", ("col", 2), ("const", 0.5, np.float64)),
    "dbl_nan_eq": ("eq", ("col", 2), ("const", float("nan"), np.float64)),
    "dbl_ge_nan": ("ge", ("col", 2), ("const", float("nan"), np.float64)),
    "dbl_lt_nan": ("lt", ("col", 2), ("const", float("nan"), np.float64)),
    "dbl_eq_zero": ("eq", ("col", 2), ("const", 0.0, np.float64)),
    "not_lt": ("not", ("lt", ("col", 0), ("col", 1))),
    "big": ("gt", ("col", 3), ("const", 2305843009213693952, np.int64)),
}


def filter_cols(g):
    return [(g["a"], g["a_valid"]), (g["b"], g["b_valid"]), (g["d"], g["d_valid"]), (g["e"], None)]


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_filter_golden(name):
    g = golden("filter_cases.npz")
    sel, _ = P.filter_select(FILTERS[name], filter_cols(g), len(g["a"]))
    np.testing.assert_array_equal(sel, g["sel_" + name])


def test_projection_golden():
    g = golden("filter_cases.npz")
    cols = filter_cols(g)
    n = len(g["a"])
    sel, _ = P.filter_select(FILTERS["lt_const"], cols, n)
    v, valid = P.eval_expr(("add", np.int32, ("col", 0), ("col", 1), 1), cols, n)
    np.testing.assert_array_equal(valid[sel], g["proj_add_valid"])
    np.testing.assert_array_equal(v[sel][valid[sel]], g["proj_add"][g["proj_add_valid"]])


def test_config1_golden():
    g = golden("tpch_sf001.npz")
    n = len(g["l_shipdate"])
    sel, _ = P.filter_select(("lt", ("col", 0), ("const", int(g["cfg1_date_const"].item()), np.int32)),
                             [(g["l_shipdate"], None)], n)
    assert len(sel) == 16721  # SURVEY.md section 0
    np.testing.assert_array_equal(g["l_quantity"][sel], g["cfg1_quantity"])
    assert int(g["l_quantity"][sel].sum()) == 42713700


def q1_inputs(g):
    keep = g["l_shipdate"] <= int(g["q1_date_const"].item())
    price, disc, tax = g["l_extendedprice"][keep], g["l_discount"][keep], g["l_tax"][keep]
    disc_price = price * (100 - disc)
    charge = disc_price * (100 + tax)
    return {
        "rf": g["l_returnflag"][keep], "ls": g["l_linestatus"][keep], "qty": g["l_quantity"][keep], "price": price,
        "disc": disc, "disc_price": disc_price, "charge": charge,
    }


def test_q1_golden():
    g = golden("tpch_sf001.npz")
    q = q1_inputs(g)
    n = len(q["rf"])
    res = P.group_by([(q["rf"], None), (q["ls"], None)],
                     [("sum", (q["qty"], None)), ("sum", (q["price"], None)), ("sum", (q["disc_price"], None)),
                      ("sum", (q["charge"], None)), ("avg", (q["qty"], None)), ("avg", (q["price"], None)),
                      ("avg", (q["disc"], None)), ("count_star", None)], n)
    assert len(res) == len(g["q1_returnflag"])
    for i in range(len(g["q1_returnflag"])):
        r = res[(int(g["q1_returnflag"][i]), int(g["q1_linestatus"][i]))]
        assert r[0] == int(g["q1_sum_qty_str"][i])
        assert r[1] == int(g["q1_sum_base_price_str"][i])
        assert r[2] == int(g["q1_sum_disc_price_str"][i])
        assert r[3] == int(g["q1_sum_charge_str"][i])
        # avg(DECIMAL(15,2)) in the reference divides by count*10^scale; the port returns the unscaled quotient
        assert r[4] / 100.0 == pytest.approx(float(g["q1_avg_qty"][i]), rel=1e-12)
        assert r[5] / 100.0 == pytest.approx(float(g["q1_avg_price"][i]), rel=1e-12)
        assert r[6] / 100.0 == pytest.approx(float(g["q1_avg_disc"][i]), rel=1e-12)
        assert r[7] == int(g["q1_count"][i])


def test_join_golden():
    g = golden("join_cases.npz")
    nb, npb = len(g["bk"]), len(g["pk"])
    bk, pk = [(g["bk"], g["bk_valid"])], [(g["pk"], g["pk_valid"])]
    pairs = P.hash_join(bk, pk, nb, npb, "inner")
    got = sorted((p, int(g["bp"][b])) for p, b in pairs)
    assert got == sorted(zip(g["inner_id"].tolist(), g["inner_p"].tolist()))
    left = P.hash_join(bk, pk, nb, npb, "left")
    got = sorted((p, (int(g["bp"][b]) if b >= 0 else None)) for p, b in left)
    exp = sorted(((i, (int(p) if v else None)) for i, p, v in zip(g["left_id"].tolist(), g["left_p"], g["left_p_valid"])),
                 key=lambda t: (t[0], t[1] is None, t[1] or 0))
    got = sorted(got, key=lambda t: (t[0], t[1] is None, t[1] or 0))
    assert got == exp
    assert P.hash_join(bk, pk, nb, npb, "semi") == g["semi_id"].tolist()
    assert P.hash_join(bk, pk, nb, npb, "anti") == g["anti_id"].tolist()
    m, mv = P.hash_join(bk, pk, nb, npb, "mark")
    np.testing.assert_array_equal(mv, g["mark_valid"])
    np.testing.assert_array_equal(m[mv], g["mark"][g["mark_valid"]].astype(bool))
    pairs2 = P.hash_join(bk + [(g["b2"], None)], pk + [(g["p2"], None)], nb, npb, "inner")
    got = sorted((p, int(g["bp"][b])) for p, b in pairs2)
    assert got == sorted(zip(g["inner2_id"].tolist(), g["inner2_p"].tolist()))


def test_radix_partition_ids():
    h = np.array([0, 1 << 45, 7 << 45, (1 << 48) - 1, 0xFFFF000000000000], dtype=np.uint64)
    np.testing.assert_array_equal(P.radix_partition_ids(h, 3), [0, 1, 7, 7, 0])
    np.testing.assert_array_equal(P.radix_partition_ids(h, 0), [0, 0, 0, 0, 0])


PG_GROUPBY_SQL = ("SELECT k1, k2, sum(x), count(x), count(*), min(x), max(x), avg(x), sum(d), min(d) FROM pg "
                  "GROUP BY k1, k2")


def pg_table():
    rng = np.random.default_rng(7)
    n = 4000
    k1 = rng.integers(-3, 3, size=n).astype(np.int32)
    k1v = rng.random(n) > 0.1
    k2 = rng.integers(0, 4, size=n).astype(np.uint8)
    x = rng.integers(-10 ** 12, 10 ** 12, size=n).astype(np.int64)
    xv = rng.random(n) > 0.2
    d = rng.standard_normal(n)
    return {"k1": (k1, k1v), "k2": k2, "x": (x, xv), "d": d}


def test_port_vs_live_reference_hash_and_groupby():
    """hash(k1, k2) and a GROUP BY of the port against the reference's answers on the same rows (pg_table)."""
    t = pg_table()
    (k1, k1v), k2, (x, xv), d = t["k1"], t["k2"], t["x"], t["d"]
    n = len(k2)
    want = reference_answers("port_groupby")
    assert digest(P.hash_columns([(k1, k1v), (k2, None)])) == want["hash"]
    rows = [tuple(r) for r in want["rows"]]
    res = P.group_by([(k1, k1v), (k2, None)],
                     [("sum", (x, xv)), ("count", (x, xv)), ("count_star", None), ("min", (x, xv)),
                      ("max", (x, xv)), ("avg", (x, xv)), ("sum", (d, None)), ("min", (d, None))], n)
    assert len(rows) == len(res)
    for r in rows:
        got = res[(r[0], r[1])]
        assert got[0] == r[2] and got[1] == r[3] and got[2] == r[4] and got[3] == r[5] and got[4] == r[6]
        assert got[5] == r[7] or got[5] == pytest.approx(r[7], rel=1e-15)
        assert got[6] == pytest.approx(r[8], rel=1e-9, abs=1e-9)
        assert got[7] == r[9]


JOIN_KEYS_SQL = ["jp.k = jb.k", "jp.k = jb.k AND jp.k2 = jb.k2"]
FLOAT_JOIN_KEYS = (np.array([0.0, np.nan, 1.5, -0.0, 2.5], dtype=np.float64),
                   np.array([-0.0, np.nan, 1.5, 7.0, np.nan], dtype=np.float64))


def join_tables():
    rng = np.random.default_rng(11)
    nb, npr = 700, 1500
    bk = rng.integers(0, 200, size=nb).astype(np.int64)
    bkv = rng.random(nb) > 0.05
    bk2 = rng.integers(0, 3, size=nb).astype(np.int16)
    pk = rng.integers(0, 260, size=npr).astype(np.int64)
    pkv = rng.random(npr) > 0.05
    pk2 = rng.integers(0, 3, size=npr).astype(np.int16)
    return ({"k": (bk, bkv), "k2": bk2, "id": np.arange(nb, dtype=np.int32)},
            {"k": (pk, pkv), "k2": pk2, "id": np.arange(npr, dtype=np.int32)})


def join_digest(rows):
    """canonical form of a join result: sorted (probe id, build id or -1) pairs, or sorted probe ids"""
    return digest(np.array(sorted(rows), dtype=np.int64))


def test_port_vs_live_reference_joins():
    """every join type of the port against the reference's answers (join_tables): NULL keys on both sides,
    duplicate build keys, composite keys, float keys with NaN / -0.0."""
    jb, jp = join_tables()
    nb, npr = len(jb["id"]), len(jp["id"])
    bk, bkv = jb["k"]
    pk, pkv = jp["k"]
    want = reference_answers("port_joins")
    for i, (bkeys, pkeys) in enumerate([([(bk, bkv)], [(pk, pkv)]),
                                        ([(bk, bkv), (jb["k2"], None)], [(pk, pkv), (jp["k2"], None)])]):
        assert join_digest(P.hash_join(bkeys, pkeys, nb, npr, "inner")) == want[f"inner{i}"]
        assert join_digest(P.hash_join(bkeys, pkeys, nb, npr, "left")) == want[f"left{i}"]
        assert join_digest(P.hash_join(bkeys, pkeys, nb, npr, "semi")) == want[f"semi{i}"]
        assert join_digest(P.hash_join(bkeys, pkeys, nb, npr, "anti")) == want[f"anti{i}"]
    # MARK join = `k IN (subquery)` in the select list: TRUE / FALSE / NULL (-1) per probe row
    matched, valid = P.hash_join([(bk, bkv)], [(pk, pkv)], nb, npr, "mark")
    assert digest(np.where(valid, np.asarray(matched).astype(bool), -1).astype(np.int64)) == want["mark"]
    # float keys: NaN joins NaN, -0.0 joins +0.0 (comparison_operators.cpp:24-40)
    fb, fp = FLOAT_JOIN_KEYS
    got = P.hash_join([(fb, None)], [(fp, None)], len(fb), len(fp), "inner")
    assert got == sorted(tuple(r) for r in want["float_inner"])


def fl_table():
    rng = np.random.default_rng(13)
    n = 3000
    a = rng.integers(-5, 6, size=n).astype(np.int32)
    av = rng.random(n) > 0.15
    b = rng.integers(-5, 6, size=n).astype(np.int32)
    bv = rng.random(n) > 0.15
    f = rng.choice(np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 1.5, -2.25]), size=n)
    fv = rng.random(n) > 0.1
    g = rng.choice(np.array([np.nan, np.inf, -0.0, 0.0, 1.5, 3.0]), size=n)
    return {"id": np.arange(n, dtype=np.int32), "a": (a, av), "b": (b, bv), "f": (f, fv), "g": g}


_A, _B, _F, _G = ("col", 0), ("col", 1), ("col", 2), ("col", 3)
_C3 = ("const", 3, np.int32)
FL_CASES = {   # WHERE clause -> the port's predicate over (a, b, f, g)
    "a < b": ("lt", _A, _B),
    "a = b OR a > 3": ("or", ("eq", _A, _B), ("gt", _A, _C3)),
    "a <> b AND b <= 3": ("and", ("ne", _A, _B), ("le", _B, _C3)),
    "NOT (a >= b)": ("not", ("ge", _A, _B)),
    "a IS NULL OR b IS NOT NULL": ("or", ("isnull", _A), ("isnotnull", _B)),
    "a IS DISTINCT FROM b": ("distinct", _A, _B),
    "a IS NOT DISTINCT FROM b": ("notdistinct", _A, _B),
    "(a < b) IS NULL": ("isnull", ("lt", _A, _B)),
    "NOT (a < b AND b < 3) OR a = 3": ("or", ("not", ("and", ("lt", _A, _B), ("lt", _B, _C3))), ("eq", _A, _C3)),
    "f < g": ("lt", _F, _G),
    "f >= g": ("ge", _F, _G),
    "f = g": ("eq", _F, _G),
    "f <> g": ("ne", _F, _G),
    "f IS NOT DISTINCT FROM g": ("notdistinct", _F, _G),
    "f > 1.5::DOUBLE": ("gt", _F, ("const", 1.5, np.float64)),
}


def test_port_vs_live_reference_filters():
    """three-valued logic, NULL comparisons, IS [NOT] DISTINCT FROM and the float total order of the port against
    the reference's WHERE clause, on random data with NULLs / NaN / infinities (fl_table)."""
    t = fl_table()
    n = len(t["id"])
    cols = [t["a"], t["b"], t["f"], (t["g"], None)]
    want = reference_answers("port_filters")
    assert set(want) == set(FL_CASES)
    for sql, tree in FL_CASES.items():
        sel, _ = P.filter_select(tree, cols, n)
        assert join_digest(sel.tolist()) == want[sql], sql


def test_aggregate_kats_from_reference_tests():
    """Known answers of the reference's own aggregate tests, replayed through the port:
    test/sql/aggregate/aggregates/test_sum.test:6-62 (int sums incl. the hugeint result of 1000 values near 2^62,
    all-NULL -> NULL) and test_bigint_avg.test:5-17 (AVG over integers needs the long-double finalisation:
    (2^53 + 1 + 0) / 3 = 3002399751580331 exactly)."""
    def one_group(func, values, valid=None):
        n = len(values)
        res = P.group_by([(np.zeros(n, dtype=np.int8), None)], [(func, (values, valid))], n)
        return res[(0,)][0]

    ints = np.arange(0, 1000, dtype=np.int32)
    assert one_group("sum", ints) == 499500
    both = np.concatenate([ints, np.arange(0, -1000, -1, dtype=np.int32)])
    assert one_group("sum", both) == 0
    more = np.concatenate([both, np.arange(0, -1000, -1, dtype=np.int32)])
    assert one_group("sum", more) == -499500
    assert one_group("sum", np.full(3000, -1, dtype=np.int32)) == -3000
    assert one_group("sum", ints, np.zeros(1000, dtype=bool)) is None          # no (valid) values -> NULL
    big = np.arange(4611686018427387904, 4611686018427388904, dtype=np.int64)
    assert one_group("sum", big) == 4611686018427388403500                       # needs 128 bits
    assert one_group("sum_no_overflow", np.array([5, 7], dtype=np.int64)) == 12
    avg = one_group("avg", np.array([9007199254740992, 1, 0], dtype=np.int64))
    assert avg - 3002399751580331.0 == 0.0
    assert one_group("count", ints, ints % 2 == 0) == 500
    assert one_group("min", both) == -999 and one_group("max", both) == 999


def test_join_kats_from_reference_tests():
    """Known answers of the reference's own join tests, replayed through the port:
    test/sql/join/inner/test_join.test:9-26 (duplicate build keys), left_outer/test_left_outer.test:8-24
    (unmatched probe row -> NULL payload), semianti/semijoin.test:6-62 and antijoin.test (probe rows are not
    deduplicated, build duplicates do not multiply them)."""
    i32 = np.int32
    # test (a, b) x test2 (b, c) on b
    a, tb = np.array([11, 12, 13], dtype=i32), np.array([1, 2, 3], dtype=i32)
    t2b, c = np.array([1, 1, 2], dtype=i32), np.array([10, 20, 30], dtype=i32)
    pairs = P.hash_join([(t2b, None)], [(tb, None)], 3, 3, "inner")
    assert sorted((int(a[p]), int(tb[p]), int(c[b])) for p, b in pairs) == [(11, 1, 10), (11, 1, 20), (12, 2, 30)]
    # integers (i, j) LEFT JOIN integers2 (k, l) on i = k
    i, j = np.array([1, 2, 3], dtype=i32), np.array([2, 3, 4], dtype=i32)
    k, l = np.array([1, 2], dtype=i32), np.array([10, 20], dtype=i32)
    left = P.hash_join([(k, None)], [(i, None)], 2, 3, "left")
    rows = [(int(i[p]), int(j[p]), None if b < 0 else int(k[b]), None if b < 0 else int(l[b])) for p, b in left]
    assert sorted(rows, key=lambda r: r[0]) == [(1, 2, 1, 10), (2, 3, 2, 20), (3, 4, None, None)]
    # left_table (a, b, c) SEMI / ANTI JOIN right_table (a, b) on a
    la = np.array([42, 43, 42, 42, 42, 42], dtype=i32)
    lc = np.array([1, 1, 5, 5, 5, 5], dtype=i32)
    ra = np.array([42], dtype=i32)
    semi = P.hash_join([(ra, None)], [(la, None)], 1, 6, "semi")
    assert sorted((int(la[p]), int(lc[p])) for p in semi) == [(42, 1), (42, 5), (42, 5), (42, 5), (42, 5)]
    la2 = np.array([42, 43, 43, 43, 43, 43], dtype=i32)
    anti = P.hash_join([(ra, None)], [(la2, None)], 1, 6, "anti")
    assert sorted((int(la2[p]), int(lc[p])) for p in anti) == [(43, 1), (43, 5), (43, 5), (43, 5), (43, 5)]
    # a duplicated build key does not duplicate SEMI results
    assert P.hash_join([(np.array([42, 42], dtype=i32), None)], [(la, None)], 2, 6, "semi") == semi


def test_filter_kats_from_reference_tests():
    """test/sql/filter/test_expression_executor_select.test replayed through the port (the VARCHAR values are
    replaced by their order-preserving codes duck=0 < goose=1 < swan=2): constant = constant selects all or
    nothing, NULL IS NOT DISTINCT FROM NULL is TRUE, `s = const` drops the NULL row, IS NOT DISTINCT FROM NULL
    selects exactly the NULL row, BETWEEN is two comparisons."""
    n = 6
    ids = np.arange(1, 7, dtype=np.int32)
    s = np.array([0, 1, 0, 0, 2, 0], dtype=np.int32)
    sv = np.array([True, True, False, True, True, True])
    cols = [(ids, None), (s, sv)]
    S = ("col", 1)

    def const(v, null=False):
        return ("const", 0 if null else v, np.int32, null)

    def ids_where(pred):
        sel, _ = P.filter_select(pred, cols, n)
        return ids[sel].tolist()

    assert len(ids_where(("eq", const(1), const(1)))) == 6
    assert ids_where(("eq", const(1), const(2))) == []
    assert len(ids_where(("notdistinct", const(0, True), const(0, True)))) == 6
    assert ids_where(("notdistinct", const(1), const(0, True))) == []
    assert ids_where(("eq", S, const(0))) == [1, 4, 6]
    assert ids_where(("eq", S, const(1))) == [2]
    assert ids_where(("notdistinct", S, const(0, True))) == [3]
    assert ids_where(("notdistinct", S, const(0))) == [1, 4, 6]
    assert ids_where(("and", ("ge", S, const(0)), ("le", S, const(1)))) == [1, 2, 4, 6]

"""Parity of the CUDA path (through the C ABI) with the oracle, the golden fixtures of the unmodified
reference and the reference's recorded answers on seeded random rows.  Integer results bit-exact;
double SUM/AVG within 1e-9 relative (BASELINE.json north_star)."""
import numpy as np
import pytest

from conftest import digest, golden, reference_answers
from duckdb_b200 import capi
from duckdb_b200 import operators as ops
from oracle import port as P
from test_oracle import FILTERS, filter_cols, q1_inputs

pytestmark = pytest.mark.gpu

TYPE = capi.TYPE_OF_DTYPE


def dev_u64(n):
    import torch
    return torch.empty(max(n, 1), dtype=torch.int64, device="cuda:0")


def gpu_hash(ctx, vectors, n):
    b = ops.Batch.upload(ctx, vectors, n)
    out = dev_u64(n)
    ops.hash_keys(ctx, b, list(range(len(vectors))), out.data_ptr())
    ctx.sync()
    return out[:n].cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------ hash
@pytest.mark.parametrize("name", ["i8", "i16", "i32", "i64", "u8", "u16", "u32", "u64", "f32", "f64"])
def test_hash_golden(ctx, name):
    g = golden("hash_kat.npz")
    v, valid = g[f"{name}_v"], g[f"{name}_valid"]
    h = gpu_hash(ctx, [ops.Vector.flat(v, valid)], len(v))
    np.testing.assert_array_equal(h, g[f"{name}_h"])


def test_hash_multi_bool_const_dict(ctx):
    g = golden("hash_kat.npz")
    n = len(g["multi_a"])
    h = gpu_hash(ctx, [ops.Vector.flat(g["multi_a"], g["multi_a_valid"]), ops.Vector.flat(g["multi_b"], g["multi_b_valid"]),
                       ops.Vector.flat(g["multi_c"])], n)
    np.testing.assert_array_equal(h, g["multi_h"])
    np.testing.assert_array_equal(gpu_hash(ctx, [ops.Vector.flat(g["bool_v"])], len(g["bool_v"])), g["bool_h"])
    # constant and dictionary vectors hash like their flattened form
    hc = gpu_hash(ctx, [ops.Vector.constant(7, np.int32)], 100)
    np.testing.assert_array_equal(hc, P.hash_values(np.full(100, 7, dtype=np.int32)))
    hn = gpu_hash(ctx, [ops.Vector.constant(0, np.int64, is_null=True)], 10)
    assert (hn == P.NULL_HASH).all()
    rng = np.random.default_rng(1)
    d = rng.integers(-100, 100, size=50).astype(np.int64)
    dv = rng.random(50) > 0.2
    sel = rng.integers(0, 50, size=1000).astype(np.uint32)
    hd = gpu_hash(ctx, [ops.Vector.dictionary(d, sel, dv)], 1000)
    np.testing.assert_array_equal(hd, P.hash_columns([(d[sel], dv[sel])]))


def test_hash_empty(ctx):
    b = ops.Batch.upload(ctx, [ops.Vector.flat(np.zeros(0, dtype=np.int64))], 0)
    out = dev_u64(0)
    ops.hash_keys(ctx, b, [0], out.data_ptr())
    ctx.sync()


# ------------------------------------------------------------------ filter
def build_expr(e, node, types):
    """oracle tuple tree -> b200 program; returns node index."""
    op = node[0]
    if op == "col":
        return e.col(node[1], types[node[1]])
    if op == "const":
        return e.const(node[1], TYPE[np.dtype(node[2])], len(node) > 3 and node[3])
    cmpmap = {"eq": capi.EXPR_EQ, "ne": capi.EXPR_NE, "lt": capi.EXPR_LT, "gt": capi.EXPR_GT, "le": capi.EXPR_LE,
              "ge": capi.EXPR_GE, "distinct": capi.EXPR_DISTINCT, "notdistinct": capi.EXPR_NOT_DISTINCT}
    if op in cmpmap:
        return e.cmp(cmpmap[op], build_expr(e, node[1], types), build_expr(e, node[2], types))
    if op == "and":
        return e.and_(build_expr(e, node[1], types), build_expr(e, node[2], types))
    if op == "or":
        return e.or_(build_expr(e, node[1], types), build_expr(e, node[2], types))
    if op == "not":
        return e.not_(build_expr(e, node[1], types))
    if op == "isnull":
        return e.is_null(build_expr(e, node[1], types))
    if op == "isnotnull":
        return e.is_not_null(build_expr(e, node[1], types))
    if op in ("add", "sub", "mul"):
        m = {"add": capi.EXPR_ADD, "sub": capi.EXPR_SUB, "mul": capi.EXPR_MUL}[op]
        return e.arith(m, TYPE[np.dtype(node[1])], build_expr(e, node[2], types), build_expr(e, node[3], types),
                       node[4] if len(node) > 4 else 1)
    if op == "cast":
        return e.cast(build_expr(e, node[2], types), TYPE[np.dtype(node[1])])
    raise ValueError(op)


def run_filter(ctx, cols, n, pred, projs=(), vectors=None):
    vectors = vectors or [ops.Vector.flat(v, valid) for v, valid in cols]
    types = [v.type for v in vectors]
    e = ops.Expr()
    root = build_expr(e, pred, types) if pred is not None else -1
    proots = [build_expr(e, p, types) for p in projs]
    b = ops.Batch.upload(ctx, vectors, n)
    fp = ops.FilterProject(ctx, e, root, proots)
    out, count, sel, mask = fp.execute(b, want_sel=True, want_mask=pred is not None)
    outs = out.download_all() if out is not None else []
    return count, sel, mask, outs


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_filter_golden(ctx, name):
    g = golden("filter_cases.npz")
    cols = filter_cols(g)
    n = len(g["a"])
    count, sel, mask, _ = run_filter(ctx, cols, n, FILTERS[name])
    np.testing.assert_array_equal(sel, g["sel_" + name])
    assert count == len(g["sel_" + name])
    keep = np.zeros(n, dtype=bool)
    keep[g["sel_" + name]] = True
    np.testing.assert_array_equal(capi.valid_from_words(mask, n), keep)  # bit-exact filter mask
    if n % 64:
        assert int(mask[-1]) >> (n % 64) == 0


def test_filter_projection_golden(ctx):
    g = golden("filter_cases.npz")
    cols = filter_cols(g)
    n = len(g["a"])
    count, sel, _, outs = run_filter(ctx, cols, n, FILTERS["lt_const"],
                                     [("add", np.int32, ("col", 0), ("col", 1), 1), ("col", 3)])
    v, valid = outs[0]
    np.testing.assert_array_equal(valid, g["proj_add_valid"])
    np.testing.assert_array_equal(v[valid], g["proj_add"][g["proj_add_valid"]])
    np.testing.assert_array_equal(outs[1][0], g["e"][sel])


def test_config1_golden(ctx):
    """BASELINE config 1: SELECT l_quantity FROM lineitem WHERE l_shipdate < DATE '1994-01-01' (SF0.01)."""
    g = golden("tpch_sf001.npz")
    n = len(g["l_shipdate"])
    pred = ("lt", ("col", 0), ("const", int(g["cfg1_date_const"].item()), np.int32))
    count, sel, _, outs = run_filter(ctx, [(g["l_shipdate"], None), (g["l_quantity"], None)], n, pred, [("col", 1)])
    assert count == 16721
    np.testing.assert_array_equal(outs[0][0], g["cfg1_quantity"])
    assert int(outs[0][0].sum()) == 42713700


def test_filter_vector_shapes_and_sizes(ctx):
    """flat / constant / dictionary inputs, ragged sizes around the 2048-row tile and 64-bit mask words."""
    rng = np.random.default_rng(3)
    for n in [0, 1, 31, 32, 33, 63, 64, 65, 2047, 2048, 2049, 100001]:
        d = rng.integers(-10, 10, size=17).astype(np.int16)
        dv = rng.random(17) > 0.3
        sel = rng.integers(0, 17, size=max(n, 1)).astype(np.uint32)
        a = rng.integers(-10, 10, size=max(n, 1)).astype(np.int16)
        vectors = [ops.Vector.dictionary(d, sel, dv), ops.Vector.flat(a), ops.Vector.constant(3, np.int16)]
        cols = [(d[sel][:n], dv[sel][:n]), (a[:n], None), (np.full(n, 3, dtype=np.int16), None)]
        pred = ("and", ("le", ("col", 0), ("col", 1)), ("gt", ("col", 1), ("sub", np.int16, ("col", 2), ("const", 6, np.int16), 1)))
        exp_sel, keep = P.filter_select(pred, cols, n)
        count, got_sel, mask, outs = run_filter(ctx, None, n, pred, [("col", 0), ("col", 2)], vectors=vectors)
        assert count == len(exp_sel)
        np.testing.assert_array_equal(got_sel, exp_sel)
        if n:
            np.testing.assert_array_equal(capi.valid_from_words(mask, n), keep)
            np.testing.assert_array_equal(outs[0][1], cols[0][1][exp_sel])
            np.testing.assert_array_equal(outs[0][0][outs[0][1]], cols[0][0][exp_sel][outs[0][1]])
            np.testing.assert_array_equal(outs[1][0], np.full(count, 3, dtype=np.int16))


def test_projection_only_and_decimal_overflow(ctx):
    rng = np.random.default_rng(4)
    n = 5000
    price = rng.integers(90000, 10 ** 7, size=n).astype(np.int64)
    disc = rng.integers(0, 11, size=n).astype(np.int64)
    # l_extendedprice * (1 - l_discount) as DECIMAL arithmetic on int64
    expr = ("mul", np.int64, ("col", 0), ("sub", np.int64, ("const", 100, np.int64), ("col", 1), 2), 2)
    count, sel, _, outs = run_filter(ctx, [(price, None), (disc, None)], n, None, [expr])
    assert count == n
    np.testing.assert_array_equal(sel, np.arange(n, dtype=np.uint32))
    np.testing.assert_array_equal(outs[0][0], price * (100 - disc))
    big = np.full(n, 10 ** 17, dtype=np.int64)
    with pytest.raises(capi.B200Error) as e:
        run_filter(ctx, [(big, None), (disc, None)], n, None, [("mul", np.int64, ("col", 0), ("const", 100, np.int64), 2)])
    assert e.value.code == capi.ERR_OVERFLOW
    # but not for rows the filter removes (DuckDB evaluates the projection after the filter)
    count, _, _, outs = run_filter(ctx, [(big, None), (disc, None)], n, ("lt", ("col", 1), ("const", 0, np.int64)),
                                   [("mul", np.int64, ("col", 0), ("const", 100, np.int64), 2)])
    assert count == 0


# ------------------------------------------------------------------ aggregate
AGGF = {"count_star": capi.AGG_COUNT_STAR, "count": capi.AGG_COUNT, "sum": capi.AGG_SUM,
        "sum_no_overflow": capi.AGG_SUM_NO_OVERFLOW, "min": capi.AGG_MIN, "max": capi.AGG_MAX, "avg": capi.AGG_AVG}


def agg_inputs(aggs):
    """distinct aggregate input columns (by identity) -> (list of columns, per-aggregate input index)."""
    cols, index, ids = [], [], {}
    for f, c in aggs:
        if c is None:
            index.append(-1)
            continue
        k = (id(c[0]), id(c[1]))
        if k not in ids:
            ids[k] = len(cols)
            cols.append(c)
        index.append(ids[k])
    return cols, index


def run_agg(ctx, key_cols, aggs, n, batches=1, expected_groups=0, vectors=None):
    """aggs: list of (func, (values, valid)|None). Returns dict key tuple -> results like oracle.group_by."""
    in_cols, in_index = agg_inputs(aggs)
    cols = list(key_cols) + in_cols
    key_idx = list(range(len(key_cols)))
    agg_idx = [len(key_cols) + i for i in range(len(in_cols))]
    key_types = [TYPE[np.asarray(v).dtype] for v, _ in key_cols]
    descs = [(AGGF[f], TYPE[np.asarray(c[0]).dtype] if c is not None else capi.INT64, ix)
             for (f, c), ix in zip(aggs, in_index)]
    agg = ops.HashAggregate(ctx, key_types, descs, expected_groups)
    bounds = np.linspace(0, n, batches + 1).astype(np.int64)
    for i in range(batches):
        lo, hi = int(bounds[i]), int(bounds[i + 1])
        if vectors is not None:
            vs = vectors(lo, hi)
        else:
            vs = [ops.Vector.flat(np.asarray(v)[lo:hi], None if valid is None else valid[lo:hi]) for v, valid in cols]
        b = ops.Batch.upload(ctx, vs, hi - lo)
        agg.sink(b, key_idx, agg_idx)
    ngroups = agg.group_count()
    out = agg.finalize()
    res = out.download_all()
    assert out.nrows == ngroups
    table = {}
    nk = len(key_cols)
    for g in range(out.nrows):
        key = []
        for j in range(nk):
            v, valid = res[j]
            if not valid[g]:
                key.append(None)
            elif v.dtype.kind == "f":
                key.append(int(np.array([v[g]], dtype=np.float64).view(np.uint64)[0]) if v.dtype == np.float64 else
                           int(np.array([v[g]]).view(np.uint32)[0]))
            else:
                key.append(v[g].item())
        vals = []
        for a in range(len(aggs)):
            v, valid = res[nk + a]
            vals.append((v[g].item() if hasattr(v[g], "item") else v[g]) if valid[g] else None)
        assert tuple(key) not in table, "duplicate group in the output"
        table[tuple(key)] = vals
    agg.close()
    return table


def assert_groups_equal(got, exp, aggs):
    assert set(got) == set(exp)
    for k, e in exp.items():
        for (f, c), gv, ev in zip(aggs, got[k], e):
            isf = c is not None and np.asarray(c[0]).dtype.kind == "f"
            if ev is None or gv is None:
                assert gv is None and ev is None, (k, f, gv, ev)
            elif isinstance(ev, float) and np.isnan(ev):
                assert np.isnan(gv)
            elif f in ("sum", "avg") and isf:
                assert gv == pytest.approx(ev, rel=1e-9, abs=1e-12), (k, f)   # tolerance of BASELINE.json
            elif f == "avg":
                assert gv == ev or gv == pytest.approx(ev, rel=1e-15), (k, f, gv, ev)
            else:
                assert gv == ev, (k, f, gv, ev)  # bit-exact


def test_q1_golden(ctx):
    """TPC-H Q1 shape on SF0.01 against the reference's HASH_GROUP_BY answer (sums bit-exact, avgs 1e-9)."""
    g = golden("tpch_sf001.npz")
    q = q1_inputs(g)
    n = len(q["rf"])
    qty, price = (q["qty"], None), (q["price"], None)
    aggs = [("sum", qty), ("sum", price), ("sum", (q["disc_price"], None)), ("sum", (q["charge"], None)),
            ("avg", qty), ("avg", price), ("avg", (q["disc"], None)), ("count_star", None)]
    for batches in (1, 3):
        got = run_agg(ctx, [(q["rf"], None), (q["ls"], None)], aggs, n, batches=batches)
        assert len(got) == len(g["q1_returnflag"])
        for i in range(len(g["q1_returnflag"])):
            r = got[(int(g["q1_returnflag"][i]), int(g["q1_linestatus"][i]))]
            assert r[0] == int(g["q1_sum_qty_str"][i])
            assert r[1] == int(g["q1_sum_base_price_str"][i])
            assert r[2] == int(g["q1_sum_disc_price_str"][i])
            assert r[3] == int(g["q1_sum_charge_str"][i])
            assert r[4] / 100.0 == pytest.approx(float(g["q1_avg_qty"][i]), rel=1e-9)
            assert r[5] / 100.0 == pytest.approx(float(g["q1_avg_price"][i]), rel=1e-9)
            assert r[6] / 100.0 == pytest.approx(float(g["q1_avg_disc"][i]), rel=1e-9)
            assert r[7] == int(g["q1_count"][i])


def test_q3_groupby_golden(ctx):
    """Q3's 3-key group-by (i64, date i32, i32) over the golden join output: high-cardinality global path."""
    g = golden("tpch_sf001.npz")
    keep_o = g["o_orderdate"] < int(g["q3_date"].item())
    omap = {int(k): i for i, k in enumerate(g["o_orderkey"]) if keep_o[i]}
    keep_l = g["l_shipdate"] > int(g["q3_date"].item())
    rows = [i for i in np.nonzero(keep_l)[0] if int(g["l_orderkey"][i]) in omap]
    oi = np.array([omap[int(g["l_orderkey"][i])] for i in rows])
    rows = np.array(rows)
    k1, k2, k3 = g["l_orderkey"][rows], g["o_orderdate"][oi], g["o_shippriority"][oi]
    rev = g["l_extendedprice"][rows] * (100 - g["l_discount"][rows])
    got = run_agg(ctx, [(k1, None), (k2, None), (k3, None)], [("sum", (rev, None)), ("count_star", None)], len(rows),
                  batches=2)
    assert len(got) == len(g["q3_orderkey"])
    for i in range(len(g["q3_orderkey"])):
        r = got[(int(g["q3_orderkey"][i]), int(g["q3_orderdate"][i]), int(g["q3_shippriority"][i]))]
        assert r[0] == int(g["q3_revenue_str"][i]) and r[1] == int(g["q3_count"][i])


@pytest.mark.parametrize("ngroups,batches", [(1, 1), (3, 2), (8, 1), (9, 1), (40, 2), (1000, 3), (200000, 2)])
def test_agg_random_vs_oracle(ctx, ngroups, batches):
    """all aggregate functions x NULL keys x NULL inputs; cardinalities straddling the fast-path directory
    (<= 8 groups), its overflow (9, 40) and table growth (200000 > initial capacity/2)."""
    rng = np.random.default_rng(ngroups)
    n = 300000 if ngroups >= 1000 else 50000
    k1 = rng.integers(0, max(1, ngroups // 3 + 1), size=n).astype(np.int32)
    k1v = rng.random(n) > 0.05
    k2 = rng.integers(0, 3, size=n).astype(np.uint8)
    x = rng.integers(-2 ** 62, 2 ** 62, size=n).astype(np.int64)   # forces 128-bit carries
    xv = rng.random(n) > 0.3
    y = rng.integers(0, 1000, size=n).astype(np.int16)
    d = rng.standard_normal(n) * 1e6
    dv = rng.random(n) > 0.1
    f = rng.standard_normal(n).astype(np.float32)
    u = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    xc, yc, dc = (x, xv), (y, None), (d, dv)
    aggs = [("sum", xc), ("count", xc), ("count_star", None), ("min", xc), ("max", xc), ("avg", xc),
            ("sum_no_overflow", yc), ("sum", dc), ("avg", dc), ("min", dc), ("max", (f, None)), ("sum", (u, None)),
            ("min", yc)]
    keys = [(k1, k1v), (k2, None)]
    exp = P.group_by(keys, aggs, n)
    got = run_agg(ctx, keys, aggs, n, batches=batches)
    assert_groups_equal(got, exp, aggs)


@pytest.mark.parametrize("g1,g2", [(3, 2), (7, 5), (40, 50), (3000, 1000)])
def test_agg_paths_large(ctx, g1, g2):
    """> 2 M rows so that the adaptive path selection runs: register FAST (6 groups), MID (35 / 2000 groups),
    GLOBAL with table growth (3 M groups).  Checked against vectorised numpy sums (exact integers)."""
    rng = np.random.default_rng(g1 * 7 + g2)
    n = 5_000_000 + 777
    kdt = np.uint8 if g1 < 256 else np.int32
    k1 = rng.integers(0, g1, size=n).astype(kdt)
    k2 = rng.integers(0, g2, size=n).astype(kdt)
    a = rng.integers(-10 ** 9, 10 ** 9, size=n).astype(np.int64)
    b = rng.integers(0, 10 ** 7, size=n).astype(np.int64)
    b[::1000003] = 2 ** 50            # "big" values: must leave the register fast path, result still exact
    c = rng.integers(0, 100, size=n).astype(np.int32)
    ac, bc, cc = (a, None), (b, None), (c, None)
    aggs = [("sum", ac), ("sum", bc), ("avg", ac), ("sum_no_overflow", cc), ("count", cc), ("count_star", None)]
    got = run_agg(ctx, [(k1, None), (k2, None)], aggs, n, batches=2)
    gid = k1.astype(np.int64) * g2 + k2
    ng = g1 * g2
    cnt = np.bincount(gid, minlength=ng)
    sa = np.zeros(ng, dtype=np.int64)
    sb = np.zeros(ng, dtype=np.int64)
    sc = np.zeros(ng, dtype=np.int64)
    np.add.at(sa, gid, a)
    np.add.at(sb, gid, b)
    np.add.at(sc, gid, c.astype(np.int64))
    present = np.nonzero(cnt)[0]
    assert len(got) == len(present)
    for g in present[:: max(1, len(present) // 5000)]:
        r = got[(int(g // g2), int(g % g2))]
        assert r[0] == int(sa[g]) and r[1] == int(sb[g]) and r[3] == int(sc[g]) and r[4] == int(cnt[g]) and r[5] == int(cnt[g])
        assert r[2] == float(np.longdouble(int(sa[g])) / np.longdouble(int(cnt[g])))
    assert sum(v[5] for v in got.values()) == n


@pytest.mark.parametrize("g1,g2,nsum,knob", [(7, 5, 1, None), (7, 5, 5, None), (11, 5, 2, None), (16, 8, 1, None),
                                             (25, 10, 3, None), (25, 24, 1, None), (7, 5, 1, "B200_AGG_NO_WPRIV"),
                                             (7, 5, 5, "B200_AGG_NO_WPRIV"), (7, 5, 1, "B200_AGG_WPRIV"), (7, 5, 2, "B200_AGG_NO_DIRECT"),
                                             (16, 8, 1, "B200_AGG_NO_DIRECT")])
def test_agg_priv_path(ctx, monkeypatch, g1, g2, nsum, knob):
    """9..600 groups of 8-byte integer sums through agg_priv.cu: warp-private accumulators with match.any rounds
    (WPRIV, direct slot tables), thread-private accumulators (B200_AGG_NO_WPRIV) and the directory lookup
    (B200_AGG_NO_DIRECT); shapes beyond a path's slots overflow into the global table / fall back to MID.  Includes
    values beyond +-2^40 (global path inline) and negative values.  Exact against numpy integer sums."""
    if knob:
        monkeypatch.setenv(knob, "1")
    rng = np.random.default_rng(g1 * 31 + g2 + nsum)
    n = 4_500_000 + 333
    k1 = rng.integers(0, g1, size=n).astype(np.uint8)
    k2 = rng.integers(0, g2, size=n).astype(np.uint8)
    cols = [rng.integers(-10 ** 9, 10 ** 10, size=n).astype(np.int64) for _ in range(nsum)]
    cols[0][::700001] = -(2 ** 55)
    aggs = [("sum", (c, None)) for c in cols] + [("avg", (cols[0], None)), ("count_star", None)]
    got = run_agg(ctx, [(k1, None), (k2, None)], aggs, n, batches=2)
    gid = k1.astype(np.int64) * g2 + k2
    ng = g1 * g2
    cnt = np.bincount(gid, minlength=ng)
    assert len(got) == int((cnt > 0).sum())
    for j, c in enumerate(cols):
        # exact 128-bit reference: split into 32-bit halves so that np.add.at cannot overflow
        lo = np.zeros(ng, dtype=np.int64)
        hi = np.zeros(ng, dtype=np.int64)
        np.add.at(lo, gid, (c & 0xffffffff).astype(np.int64))
        np.add.at(hi, gid, c >> 32)
        for g in np.nonzero(cnt)[0]:
            assert got[(int(g // g2), int(g % g2))][j] == (int(hi[g]) << 32) + int(lo[g]), (g, j)
    assert sum(v[-1] for v in got.values()) == n


def test_agg_float_keys_nan_zero_and_all_null_inputs(ctx):
    n = 4000
    rng = np.random.default_rng(9)
    k = rng.choice(np.array([0.0, -0.0, np.nan, -np.nan, 1.5, np.inf]), size=n)
    x = rng.integers(-100, 100, size=n).astype(np.int32)
    xv = np.zeros(n, dtype=bool)  # every input NULL -> SUM/MIN/AVG are NULL, COUNT is 0
    xc = (x, xv)
    aggs = [("sum", xc), ("min", xc), ("avg", xc), ("count", xc), ("count_star", None)]
    exp = P.group_by([(k, None)], aggs, n)
    got = run_agg(ctx, [(k, None)], aggs, n)
    assert len(got) == 4  # {0.0, NaN, 1.5, inf}
    assert_groups_equal(got, exp, aggs)


def test_agg_const_and_dict_vectors(ctx):
    rng = np.random.default_rng(11)
    n = 30000
    d = np.array([10, 20, 30, 40], dtype=np.int64)
    dv = np.array([True, True, False, True])
    sel = rng.integers(0, 4, size=n).astype(np.uint32)
    x = rng.integers(0, 100, size=n).astype(np.int64)

    def vectors(lo, hi):
        return [ops.Vector.dictionary(d, sel[lo:hi], dv), ops.Vector.constant(5, np.int8), ops.Vector.flat(x[lo:hi])]

    aggs = [("sum", (x, None)), ("count_star", None)]
    keys = [(d[sel], dv[sel]), (np.full(n, 5, dtype=np.int8), None)]
    exp = P.group_by(keys, aggs, n)
    got = run_agg(ctx, keys, aggs, n, batches=2, vectors=vectors)
    assert_groups_equal(got, exp, aggs)


def test_agg_empty_input(ctx):
    got = run_agg(ctx, [(np.zeros(0, dtype=np.int32), None)], [("count_star", None)], 0)
    assert got == {}


def test_agg_export_combine_roundtrip(ctx):
    """partial tables on two 'ranks' merged through export_states/combine_states == one table over all rows
    (GroupedAggregateHashTable::Combine, aggregate_hashtable.cpp:1168-1197)."""
    rng = np.random.default_rng(13)
    n = 40000
    k = rng.integers(0, 500, size=n).astype(np.int64)
    kv = rng.random(n) > 0.02
    x = rng.integers(-2 ** 62, 2 ** 62, size=n).astype(np.int64)
    xv = rng.random(n) > 0.2
    d = rng.standard_normal(n)
    xc, dc = (x, xv), (d, None)
    aggs = [("sum", xc), ("avg", xc), ("min", xc), ("max", dc), ("sum", dc), ("count", xc), ("count_star", None)]
    in_cols, in_index = agg_inputs(aggs)
    descs = [(AGGF[f], TYPE[np.asarray(c[0]).dtype] if c is not None else capi.INT64, ix)
             for (f, c), ix in zip(aggs, in_index)]
    parts = []
    for lo, hi in [(0, n // 3), (n // 3, n)]:
        a = ops.HashAggregate(ctx, [capi.INT64], descs)
        b = ops.Batch.upload(ctx, [ops.Vector.flat(k[lo:hi], kv[lo:hi]), ops.Vector.flat(x[lo:hi], xv[lo:hi]),
                                   ops.Vector.flat(d[lo:hi])], hi - lo)
        a.sink(b, [0], [1, 2])
        parts.append(a)
    final = ops.HashAggregate(ctx, [capi.INT64], descs)
    for a in parts:
        st = a.export_states()
        final.combine_states(st)
    out = final.finalize()
    res = out.download_all()
    exp = P.group_by([(k, kv)], aggs, n)
    got = {}
    for g in range(out.nrows):
        key = (res[0][0][g].item() if res[0][1][g] else None,)
        got[key] = [(res[1 + a][0][g].item() if hasattr(res[1 + a][0][g], "item") else res[1 + a][0][g])
                    if res[1 + a][1][g] else None for a in range(len(aggs))]
    assert_groups_equal(got, exp, aggs)


# ------------------------------------------------------------------ join
JT = {"inner": capi.JOIN_INNER, "left": capi.JOIN_LEFT, "semi": capi.JOIN_SEMI, "anti": capi.JOIN_ANTI,
      "mark": capi.JOIN_MARK}


def run_join(ctx, jt, build_keys, build_payload, probe_keys, probe_lhs, nb, npb, build_batches=1):
    """-> list of result columns [(values, valid)...] ordered [lhs..., payload... | mark]."""
    import torch
    kt = [TYPE[np.asarray(v).dtype] for v, _ in build_keys]
    pt = [TYPE[np.asarray(v).dtype] for v, _ in build_payload]
    j = ops.HashJoin(ctx, JT[jt], kt, pt)
    bounds = np.linspace(0, nb, build_batches + 1).astype(np.int64)
    for i in range(build_batches):
        lo, hi = int(bounds[i]), int(bounds[i + 1])
        vs = [ops.Vector.flat(np.asarray(v)[lo:hi], None if valid is None else valid[lo:hi])
              for v, valid in list(build_keys) + list(build_payload)]
        b = ops.Batch.upload(ctx, vs, hi - lo)
        j.sink(b, list(range(len(build_keys))), list(range(len(build_keys), len(build_keys) + len(build_payload))))
    j.finalize()
    assert j.build_rows() == nb
    vs = [ops.Vector.flat(v, valid) for v, valid in list(probe_keys) + list(probe_lhs)]
    pb = ops.Batch.upload(ctx, vs, npb)
    sel_t = torch.empty(max(1, npb * 8), dtype=torch.int32, device="cuda:0")
    out, count = j.execute(pb, list(range(len(probe_keys))),
                           list(range(len(probe_keys), len(probe_keys) + len(probe_lhs))), 0, sel_t.data_ptr())
    res = out.download_all()
    sel = sel_t[:count].cpu().numpy().view(np.uint32)
    j.close()
    return res, sel, count


def test_join_golden(ctx):
    g = golden("join_cases.npz")
    nb, npb = len(g["bk"]), len(g["pk"])
    ids = np.arange(npb, dtype=np.int32)
    bk, pk = [(g["bk"], g["bk_valid"])], [(g["pk"], g["pk_valid"])]
    res, sel, count = run_join(ctx, "inner", bk, [(g["bp"], None)], pk, [(ids, None)], nb, npb, build_batches=2)
    assert count == len(g["inner_id"])
    assert sorted(zip(res[0][0].tolist(), res[1][0].tolist())) == sorted(zip(g["inner_id"].tolist(), g["inner_p"].tolist()))
    np.testing.assert_array_equal(res[0][0], ids[sel])  # lhs_sel consistent with the gathered lhs column
    res, _, count = run_join(ctx, "left", bk, [(g["bp"], None)], pk, [(ids, None)], nb, npb)
    got = sorted(((i, (int(p) if v else None)) for i, p, v in zip(res[0][0].tolist(), res[1][0], res[1][1])),
                 key=lambda t: (t[0], t[1] is None, t[1] or 0))
    exp = sorted(((i, (int(p) if v else None)) for i, p, v in zip(g["left_id"].tolist(), g["left_p"], g["left_p_valid"])),
                 key=lambda t: (t[0], t[1] is None, t[1] or 0))
    assert got == exp
    res, _, _ = run_join(ctx, "semi", bk, [], pk, [(ids, None)], nb, npb)
    assert sorted(res[0][0].tolist()) == g["semi_id"].tolist()
    res, _, _ = run_join(ctx, "anti", bk, [], pk, [(ids, None)], nb, npb)
    assert sorted(res[0][0].tolist()) == g["anti_id"].tolist()
    res, _, count = run_join(ctx, "mark", bk, [], pk, [(ids, None)], nb, npb)
    assert count == npb
    order = np.argsort(res[0][0])
    mv = res[1][1][order]
    np.testing.assert_array_equal(mv, g["mark_valid"])
    np.testing.assert_array_equal(res[1][0][order][mv].astype(bool), g["mark"][g["mark_valid"]].astype(bool))
    # composite key
    res, _, count = run_join(ctx, "inner", bk + [(g["b2"], None)], [(g["bp"], None)], pk + [(g["p2"], None)],
                             [(ids, None)], nb, npb)
    assert sorted(zip(res[0][0].tolist(), res[1][0].tolist())) == sorted(zip(g["inner2_id"].tolist(), g["inner2_p"].tolist()))


@pytest.mark.parametrize("no_dense", [False, True])
def test_q14_join_golden(ctx, monkeypatch, no_dense):
    """TPC-H Q14 join on SF0.01: part (unique BIGINT key, UTINYINT promo payload -> inline-payload table)
    probed by date-filtered lineitem; result rows and the Q14 percentage equal the reference's.
    no_dense: B200_JOIN_NO_DENSE forces the open-addressing table, so the LEAN probe runs on it as well."""
    if no_dense:
        monkeypatch.setenv("B200_JOIN_NO_DENSE", "1")
    g = golden("tpch_sf001.npz")
    keep = (g["l_shipdate"] >= int(g["q14_lo"].item())) & (g["l_shipdate"] < int(g["q14_hi"].item()))
    lk, price, disc, ok = g["l_partkey"][keep], g["l_extendedprice"][keep], g["l_discount"][keep], g["l_orderkey"][keep]
    res, _, count = run_join(ctx, "inner", [(g["p_partkey"], None)], [(g["p_promo"], None)], [(lk, None)],
                             [(ok, None), (lk, None), (price, None), (disc, None)], len(g["p_partkey"]), len(lk))
    assert count == len(g["q14_orderkey"])
    got = sorted(zip(*(r[0].tolist() for r in res)))
    exp = sorted(zip(g["q14_orderkey"].tolist(), g["q14_partkey"].tolist(), g["q14_price"].tolist(),
                     g["q14_discount"].tolist(), g["q14_promo"].tolist()))
    assert got == exp
    rev = res[2][0].astype(object) * (100 - res[3][0].astype(object))
    promo = float(100.0 * float(sum(rev[res[4][0] == 1])) / float(sum(rev)))
    assert promo == pytest.approx(float(g["q14_result"][0]), rel=1e-9)


@pytest.mark.parametrize("dtype", [np.int8, np.int16, np.int32, np.int64, np.uint8, np.uint32, np.uint64, np.float64, np.float32])
def test_join_key_types_limits_vs_oracle(ctx, dtype):
    """numeric limits per key type (test/sql/join/inner/equality_join_limits.test), duplicates, NULLs,
    INT64_MIN (the table's empty-slot sentinel), -0.0/NaN float keys."""
    rng = np.random.default_rng(5)
    if np.dtype(dtype).kind == "f":
        pool = np.array([0.0, -0.0, np.nan, 1.0, -1.0, np.inf, -np.inf, 3.5], dtype=dtype)
    else:
        info = np.iinfo(dtype)
        pool = np.array([info.min, info.max, 0, 1, 2, 3, info.max - 1, info.min + 1], dtype=dtype)
    nb, npb = 300, 2000
    bk = rng.choice(pool, size=nb)
    bkv = rng.random(nb) > 0.1
    pk = rng.choice(pool, size=npb)
    pkv = rng.random(npb) > 0.1
    bp = np.arange(nb, dtype=np.int64)
    ids = np.arange(npb, dtype=np.int64)
    exp = P.hash_join([(bk, bkv)], [(pk, pkv)], nb, npb, "inner")
    res, _, count = run_join(ctx, "inner", [(bk, bkv)], [(bp, None)], [(pk, pkv)], [(ids, None)], nb, npb)
    assert count == len(exp)
    assert sorted(zip(res[0][0].tolist(), res[1][0].tolist())) == exp


@pytest.mark.parametrize("jt", ["inner", "left", "semi", "anti", "mark"])
@pytest.mark.parametrize("dtype,payload_dtype", [(np.int32, np.uint8), (np.int64, np.int64), (np.uint16, np.int16)])
def test_join_dense_table_vs_oracle(ctx, jt, dtype, payload_dtype):
    """unique integer build keys in a small range (negative keys, gaps, NULLs) -> the direct-addressed table
    (DuckDB's perfect hash join shape, perfect_hash_join_executor.cpp:70-133); all join types vs the oracle."""
    rng = np.random.default_rng(int(np.dtype(dtype).itemsize) * 31 + len(jt))
    lo = -500 if np.dtype(dtype).kind == "i" else 10
    universe = np.arange(lo, lo + 3000).astype(dtype)
    bk = rng.permutation(universe)[:1200]
    bkv = rng.random(len(bk)) > 0.03
    bp = rng.integers(-100, 100, size=len(bk)).astype(payload_dtype)
    pk = rng.integers(lo - 50, lo + 3050, size=5000).astype(dtype)
    pkv = rng.random(len(pk)) > 0.05
    ids = np.arange(len(pk), dtype=np.int32)
    nb, npb = len(bk), len(pk)
    payload = [(bp, None)] if jt in ("inner", "left") else []
    res, _, count = run_join(ctx, jt, [(bk, bkv)], payload, [(pk, pkv)], [(ids, None)], nb, npb)
    exp = P.hash_join([(bk, bkv)], [(pk, pkv)], nb, npb, jt)
    if jt == "inner":
        assert sorted(zip(res[0][0].tolist(), res[1][0].tolist())) == sorted((p, int(bp[b])) for p, b in exp)
    elif jt == "left":
        got = sorted(((i, (int(p) if v else None)) for i, p, v in zip(res[0][0].tolist(), res[1][0], res[1][1])),
                     key=lambda t: (t[0], t[1] is None, t[1] or 0))
        want = sorted(((p, (int(bp[b]) if b >= 0 else None)) for p, b in exp), key=lambda t: (t[0], t[1] is None, t[1] or 0))
        assert got == want
    elif jt in ("semi", "anti"):
        assert sorted(res[0][0].tolist()) == exp
    else:
        order = np.argsort(res[0][0])
        np.testing.assert_array_equal(res[1][1][order], exp[1])
        np.testing.assert_array_equal(res[1][0][order][exp[1]].astype(bool), exp[0][exp[1]])


def test_join_empty_sides(ctx):
    z = np.zeros(0, dtype=np.int64)
    k = np.arange(10, dtype=np.int64)
    res, _, count = run_join(ctx, "inner", [(z, None)], [(z, None)], [(k, None)], [(k, None)], 0, 10)
    assert count == 0
    res, _, count = run_join(ctx, "anti", [(z, None)], [], [(k, None)], [(k, None)], 0, 10)
    assert count == 10
    res, _, count = run_join(ctx, "mark", [(z, None)], [], [(k, None)], [(k, None)], 0, 10)
    assert count == 10 and res[1][1].all() and not res[1][0].any()
    res, _, count = run_join(ctx, "inner", [(k, None)], [(k, None)], [(z, None)], [(z, None)], 10, 0)
    assert count == 0


@pytest.mark.parametrize("no_dense", [False, True])
def test_join_large_roundtrip_properties(ctx, monkeypatch, no_dense):
    """size-independent properties at a larger size: PK-FK probe returns exactly one row per probe row, payload
    equals f(key), checksum of gathered columns equals the input's (dense table and open addressing)."""
    if no_dense:
        monkeypatch.setenv("B200_JOIN_NO_DENSE", "1")
    rng = np.random.default_rng(17)
    nb, npb = 1 << 20, 1 << 22
    bk = rng.permutation(nb).astype(np.int64) + 1
    bp = (bk % 251).astype(np.uint8)
    pk = rng.integers(1, nb + 1, size=npb).astype(np.int64)
    price = rng.integers(0, 10 ** 7, size=npb).astype(np.int64)
    res, sel, count = run_join(ctx, "inner", [(bk, None)], [(bp, None)], [(pk, None)], [(pk, None), (price, None)], nb, npb)
    assert count == npb
    np.testing.assert_array_equal(res[2][0], (res[0][0] % 251).astype(np.uint8))
    assert int(res[1][0].astype(object).sum()) == int(price.astype(object).sum())
    assert len(np.unique(sel)) == npb


# ------------------------------------------------------------------ radix partition
@pytest.mark.parametrize("bits", [0, 1, 3, 4, 8])
def test_radix_partition(ctx, bits):
    rng = np.random.default_rng(bits)
    n = 100000
    k = rng.integers(0, 5000, size=n).astype(np.int64)
    kv = rng.random(n) > 0.05
    v = rng.integers(0, 2 ** 31, size=n).astype(np.int32)
    b = ops.Batch.upload(ctx, [ops.Vector.flat(k, kv), ops.Vector.flat(v)], n)
    out, counts = ops.radix_partition(ctx, b, [0], bits)
    ids = P.radix_partition_ids(P.hash_columns([(k, kv)]), bits)
    np.testing.assert_array_equal(counts, np.bincount(ids, minlength=1 << bits).astype(np.uint64))
    (ok, okv), (ov, _) = out.download_all()
    off = 0
    for p in range(1 << bits):
        c = int(counts[p])
        exp = sorted(zip(np.where(kv[ids == p], k[ids == p], -1).tolist(), v[ids == p].tolist()))
        got = sorted(zip(np.where(okv[off:off + c], ok[off:off + c], -1).tolist(), ov[off:off + c].tolist()))
        assert got == exp
        off += c


@pytest.mark.parametrize("bits", [0, 1, 2, 3, 4])
def test_radix_partition_fast_path(ctx, bits):
    """few partitions, flat columns without NULLs -> the fused two-pass kernels (the GPU-level shuffle)."""
    rng = np.random.default_rng(40 + bits)
    n = 300001
    k = rng.integers(-10 ** 9, 10 ** 9, size=n).astype(np.int64)
    v = rng.integers(0, 2 ** 31, size=n).astype(np.int32)
    f = rng.integers(0, 255, size=n).astype(np.uint8)
    b = ops.Batch.upload(ctx, [ops.Vector.flat(k), ops.Vector.flat(v), ops.Vector.flat(f)], n)
    out, counts = ops.radix_partition(ctx, b, [0], bits)
    ids = P.radix_partition_ids(P.hash_columns([(k, None)]), bits)
    np.testing.assert_array_equal(counts, np.bincount(ids, minlength=1 << bits).astype(np.uint64))
    (ok, _), (ov, _), (of, _) = out.download_all()
    off = 0
    for p in range(1 << bits):
        c = int(counts[p])
        exp = sorted(zip(k[ids == p].tolist(), v[ids == p].tolist(), f[ids == p].tolist()))
        got = sorted(zip(ok[off:off + c].tolist(), ov[off:off + c].tolist(), of[off:off + c].tolist()))
        assert got == exp
        off += c


@pytest.mark.parametrize("bulk", ["0", "1"])
@pytest.mark.parametrize("bits,ncols", [(1, 3), (2, 2), (3, 1), (4, 4)])
def test_radix_partition_eight_byte_columns(ctx, bits, ncols, bulk, monkeypatch):
    """the shuffle-join's shape - BIGINT key + 8-byte payload columns - takes the register-staged scatter kernel
    (B200_PART_BULK=1: runs leave shared memory as bulk-async copies)"""
    monkeypatch.setenv("B200_PART_BULK", bulk)
    rng = np.random.default_rng(70 + bits)
    n = 250007
    k = rng.integers(-10 ** 12, 10 ** 12, size=n).astype(np.int64)
    pay = [rng.integers(-2 ** 62, 2 ** 62, size=n).astype(np.int64) for _ in range(ncols - 1)]
    # the key is not the first column when there is a payload: the kernel permutes it to the front internally
    cols = (pay[:1] + [k] + pay[1:]) if pay else [k]
    key_col = 1 if pay else 0
    b = ops.Batch.upload(ctx, [ops.Vector.flat(c) for c in cols], n)
    out, counts = ops.radix_partition(ctx, b, [key_col], bits)
    ids = P.radix_partition_ids(P.hash_columns([(k, None)]), bits)
    np.testing.assert_array_equal(counts, np.bincount(ids, minlength=1 << bits).astype(np.uint64))
    got_cols = [c for c, _ in out.download_all()]
    off = 0
    for p in range(1 << bits):
        c = int(counts[p])
        exp = sorted(zip(*[col[ids == p].tolist() for col in cols]))
        got = sorted(zip(*[col[off:off + c].tolist() for col in got_cols]))
        assert got == exp
        off += c


@pytest.mark.parametrize("bulk", ["0", "1"])
@pytest.mark.parametrize("tight", [False, True])
def test_partition_scatter_dev_capacity_guard(ctx, bulk, tight, monkeypatch):
    """b200_partition_count_dev + b200_partition_scatter_dev on ONE GPU (every destination buffer is local): the rows
    of partition p land in buffer p from the given offset; with receive buffers that are too small the rows that do not
    fit are dropped AND counted and nothing is written past the capacity (the guard words stay intact)"""
    import torch

    monkeypatch.setenv("B200_PART_BULK", bulk)
    dev = torch.device("cuda", 0)
    bits, n = 2, 180003
    rng = np.random.default_rng(5)
    k = rng.integers(1, 10 ** 9, size=n).astype(np.int64)
    k[rng.random(n) < 0.5] = 4242           # a hot key: one partition much larger than the others
    v = rng.integers(-2 ** 62, 2 ** 62, size=n).astype(np.int64)
    tk, tv = torch.from_numpy(k).to(dev), torch.from_numpy(v).to(dev)
    batch = ops.Batch.wrap(ctx, [(tk.data_ptr(), capi.INT64), (tv.data_ptr(), capi.INT64)], n, keepalive=[tk, tv])
    ids = P.radix_partition_ids(P.hash_columns([(k, None)]), bits)
    want = np.bincount(ids, minlength=4)
    counts = torch.zeros(4, dtype=torch.int64, device=dev)
    ops.partition_count_dev(ctx, batch, [0], bits, counts.data_ptr())
    ctx.sync()
    np.testing.assert_array_equal(counts.cpu().numpy(), want)
    capacity = int(want.max()) // 2 + 3 if tight else int(want.max()) + 5   # odd / even starts both occur
    guard = 64
    sentinel = -0x0123456789abcdef
    bufs = [[torch.full((capacity + guard,), sentinel, dtype=torch.int64, device=dev) for _ in range(2)] for _ in range(4)]
    start = [1, 0, 3, 2]                   # write offsets inside the destination buffers (odd and even)
    offsets = torch.tensor(start + [0] * 12, dtype=torch.int64, device=dev)
    dropped = torch.zeros(1, dtype=torch.int64, device=dev)
    dst = [bufs[p][c].data_ptr() for p in range(4) for c in range(2)]
    ops.partition_scatter_dev(ctx, batch, [0], bits, dst, offsets.data_ptr(), capacity, dropped.data_ptr())
    ctx.sync()
    expect_dropped = 0
    for p in range(4):
        fit = max(0, min(int(want[p]), capacity - start[p]))
        expect_dropped += int(want[p]) - fit
        gk, gv = bufs[p][0].cpu().numpy(), bufs[p][1].cpu().numpy()
        assert (gk[capacity:] == sentinel).all() and (gv[capacity:] == sentinel).all(), "wrote past the capacity"
        assert (gk[:start[p]] == sentinel).all(), "wrote before the offset"
        got = sorted(zip(gk[start[p]:start[p] + fit].tolist(), gv[start[p]:start[p] + fit].tolist()))
        rows = sorted(zip(k[ids == p].tolist(), v[ids == p].tolist()))
        if fit == int(want[p]):
            assert got == rows
        else:
            # which rows of the partition made it is not specified; every delivered row must be one of the partition's
            from collections import Counter
            have, need = Counter(got), Counter(rows)
            assert all(need[r] >= cnt for r, cnt in have.items()) and sentinel not in [g[0] for g in got]
    assert int(dropped.item()) == expect_dropped


# ------------------------------------------------------------------ the reference's answers on seeded random rows
LR_GROUPBY_SQL = "SELECT k, sum(x), min(x), avg(d), count(*) FROM lr GROUP BY k ORDER BY k"
LR_JOIN_SQL = "SELECT count(*), sum(lr.x), sum(ld.p) FROM lr JOIN ld ON lr.k = ld.k"
LR_AVG_SAMPLE = 64   # every 64th group (in key order) keeps its AVG in the golden file


def lr_tables():
    rng = np.random.default_rng(23)
    n = 200000
    k = rng.integers(0, 20000, size=n).astype(np.int64)
    x = rng.integers(-10 ** 9, 10 ** 9, size=n).astype(np.int64)
    d = rng.standard_normal(n)
    dim = np.unique(k)[::2].astype(np.int64)
    return {"k": k, "x": x, "d": d}, {"k": dim, "p": (dim * 3).astype(np.int64)}


def test_live_reference_groupby_and_join(ctx):
    """GROUP BY (sum / min / avg / count) and an inner join against the reference's answers on the same rows:
    keys, sums, minima and counts of every group bit-exact (by digest), AVG within 1e-9 on a sample of groups."""
    lr, ld = lr_tables()
    k, x, d = lr["k"], lr["x"], lr["d"]
    n = len(k)
    want = reference_answers("gpu_groupby_join")
    aggs = [("sum", (x, None)), ("min", (x, None)), ("avg", (d, None)), ("count_star", None)]
    got = run_agg(ctx, [(k, None)], aggs, n, batches=2)
    keys = sorted(got)
    assert len(keys) == want["groups"]
    assert digest(np.array([g[0] for g in keys], dtype=np.int64)) == want["k"]
    for i, name in ((0, "sum"), (1, "min"), (3, "count")):
        assert digest(np.array([int(got[g][i]) for g in keys], dtype=np.int64)) == want[name], name
    for g, avg in zip(keys[::LR_AVG_SAMPLE], want["avg_sample"]):
        assert got[g][2] == pytest.approx(avg, rel=1e-9, abs=1e-12)
    dim, p = ld["k"], ld["p"]
    cnt, sx, sp = want["join"]
    res, _, count = run_join(ctx, "inner", [(dim, None)], [(p, None)], [(k, None)], [(x, None)], len(dim), n)
    assert count == cnt
    assert int(res[0][0].astype(object).sum()) == sx and int(res[1][0].astype(object).sum()) == sp

"""The register-accumulator aggregate (FASTREG, agg_fastreg_kernel in agg_tile.cu) against exact numpy sums.

FASTREG takes integer group keys without NULLs and sums / averages / counts over 8-byte integers.  A tile holds
THREADS x 4 rows (896 for the TPC-H Q1 shape, 768 / 640 for wider ones); consumer thread t owns the row pairs
(2t, 2t + 1) and (2t + 2 THREADS, 2t + 2 THREADS + 1).  Values with |x| >= 2^40, rows whose key the thread has not
seen yet and groups beyond the CTA's slots leave the straight-line path, so those are placed on the edges of that
mapping here: first and last row of a thread's rows, last row of a full tile, the ragged last tile."""
import numpy as np
import pytest

from test_gpu_parity import run_agg

pytestmark = pytest.mark.gpu

TILE = 896  # THREADS x 4 rows of the <NSUM <= 5, 4 slots> instantiations
PROBE = 1 << 18  # rows of b200_agg_sink's first (adaptation) launch
EDGES = [2 ** 40 - 1, -(2 ** 40 - 1), 2 ** 40, -(2 ** 40), -(2 ** 40) - 1, -(2 ** 63), 2 ** 63 - 1]


def exact(gid, ng, cols):
    """per group: count and the exact (Python int) sum of every column"""
    cnt = np.bincount(gid, minlength=ng)
    sums = []
    for c in cols:
        # split into 32-bit halves so that np.add.at cannot overflow
        lo = np.zeros(ng, dtype=np.int64)
        hi = np.zeros(ng, dtype=np.int64)
        np.add.at(lo, gid, (c & 0xffffffff).astype(np.int64))
        np.add.at(hi, gid, c >> 32)
        sums.append([(int(hi[g]) << 32) + int(lo[g]) for g in range(ng)])
    return cnt, sums


def check(ctx, keys, cols, batches=1):
    """group by `keys` (numpy integer columns), sum of every column, avg of the first, count(*)"""
    n = len(keys[0])
    aggs = [("sum", (c, None)) for c in cols] + [("avg", (cols[0], None)), ("count_star", None)]
    got = run_agg(ctx, [(k, None) for k in keys], aggs, n, batches=batches)
    uniq, gid = np.unique(np.stack([k.astype(np.int64) for k in keys], axis=1), axis=0, return_inverse=True)
    gid = gid.reshape(-1)
    cnt, sums = exact(gid, len(uniq), cols)
    assert len(got) == len(uniq)
    for g, key in enumerate(uniq):
        v = got[tuple(int(x) for x in key)]
        for j in range(len(cols)):
            assert v[j] == sums[j][g], (tuple(key), j, v[j], sums[j][g])
        avg = float(np.longdouble(sums[0][g]) / np.longdouble(int(cnt[g])))
        assert v[len(cols)] == avg or v[len(cols)] == pytest.approx(avg, rel=1e-15), (tuple(key), v[len(cols)], avg)
        assert v[len(cols) + 1] == int(cnt[g])


def q1(n):
    import torch

    import bench_data as BD

    q = BD.Gen(torch, "cuda").q1(n)
    keys = [q["rf"].cpu().numpy(), q["ls"].cpu().numpy()]
    cols = [q[k].cpu().numpy().astype(np.int64) for k in ("qty", "price", "disc_price", "charge", "disc")]
    return keys, cols


@pytest.mark.parametrize("n", [100, 895, 896, 897, PROBE - 1, PROBE + 1, PROBE + 896 * 3 + 5, 3_000_017])
@pytest.mark.parametrize("batches", [1, 3])
def test_q1_shape(ctx, n, batches):
    if batches > 1 and n < 1000:
        pytest.skip("one batch covers the small sizes")
    keys, cols = q1(n)
    check(ctx, keys, cols, batches)


def edge_rows(n):
    """row indices on the edges of the thread / tile mapping, for launches starting at row 0 and at PROBE"""
    rows = []
    for base in (0, PROBE):
        for tile in (0, 1, 7):
            t0 = base + tile * TILE
            # thread 0 (rows 0, 1, 448, 449), thread 9 (rows 18, 19, 466, 467), thread 223 (rows 446, 447, 894, 895)
            rows += [t0 + r for r in (0, 1, 448, 449, 18, 19, 466, 467, 446, 447, 894, 895)]
    rows += [n - 1, n - 2, n - 5]  # the ragged last tile
    return sorted(set(r for r in rows if 0 <= r < n))


@pytest.mark.parametrize("batches", [1, 2])
def test_q1_range_edges(ctx, batches):
    n = PROBE + 20 * TILE + 37
    keys, cols = q1(n)
    rows = edge_rows(n)
    for i, r in enumerate(rows):
        cols[i % len(cols)][r] = EDGES[i % len(EDGES)]
        cols[(i + 2) % len(cols)][r] = EDGES[(i + 3) % len(EDGES)]
    check(ctx, keys, cols, batches)


def test_range_edges_next_to_unseen_key(ctx):
    """a wide value in the same row pair as the first row of a key the thread has not seen yet"""
    n = PROBE + 10 * TILE + 3
    rng = np.random.default_rng(5)
    k1 = np.zeros(n, dtype=np.uint8)
    k2 = np.zeros(n, dtype=np.uint8)
    cols = [rng.integers(-10 ** 6, 10 ** 9, size=n).astype(np.int64) for _ in range(3)]
    for i, r in enumerate(edge_rows(n)):
        # a new key in one row of the pair, an edge value in the other (and in both, every third time)
        mate = min(r ^ 1, n - 1)
        k1[r] = 1 + i % 3
        cols[i % 3][mate] = EDGES[i % len(EDGES)]
        if i % 3 == 0:
            cols[(i + 1) % 3][r] = EDGES[(i + 4) % len(EDGES)]
    check(ctx, [k1, k2], cols)


@pytest.mark.parametrize("groups", [5, 6, 8, 9])
def test_group_counts(ctx, groups):
    """5..8 groups take 8 directory slots; 9 overflow the directory into the global table"""
    n = 2_000_003
    rng = np.random.default_rng(groups)
    g = rng.integers(0, groups, size=n)
    k1 = (g // 3).astype(np.uint8)
    k2 = (g % 3).astype(np.uint8)
    cols = [rng.integers(-10 ** 9, 10 ** 10, size=n).astype(np.int64) for _ in range(5)]
    cols[1][::100003] = 2 ** 40
    check(ctx, [k1, k2], cols, batches=2)


@pytest.mark.parametrize("nsum", [1, 6])
def test_sum_counts(ctx, nsum):
    n = 1_000_000 + 77
    rng = np.random.default_rng(nsum)
    k1 = rng.integers(0, 2, size=n).astype(np.uint8)
    k2 = rng.integers(0, 2, size=n).astype(np.uint8)
    cols = [rng.integers(-10 ** 11, 10 ** 11, size=n).astype(np.int64) for _ in range(nsum)]
    cols[-1][::65537] = -(2 ** 40) - 1
    check(ctx, [k1, k2], cols)


@pytest.mark.parametrize("dtype", [np.uint16, np.int32], ids=["2-byte key", "4-byte key"])
def test_wider_keys(ctx, dtype):
    n = 1_500_011
    rng = np.random.default_rng(3)
    k = rng.choice(np.array([7, 300, 40000, 5], dtype=np.int64), size=n).astype(dtype)
    if dtype == np.int32:
        k[::3] = -123456789
    cols = [rng.integers(-10 ** 12, 10 ** 12, size=n).astype(np.int64) for _ in range(3)]
    for i, r in enumerate(edge_rows(n)):
        cols[i % 3][r] = EDGES[i % len(EDGES)]
    check(ctx, [k], cols, batches=2)

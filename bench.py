#!/usr/bin/env python3
"""bench.py - BASELINE.json's metric on BASELINE.json's configs, one JSON line on stdout.

  python bench.py [--gpus N --steps K --warmup W]           our arm (CUDA kernels through the C ABI)
  python bench.py --dump-outputs DIR [...]                 ... and write the headline's result as DIR/<name>.npy
  python bench.py --impl reference [...]                     the reference's CPU operators (oracle/_ref)

Workloads (synthetic TPC-H / SSB-shaped columns, defined once as DuckDB SQL and restated with torch ops in
bench_data.py, so that both arms see the same rows; row i of rank r is row i + r * n of the formulas):
  agg      (headline, configs[1]) TPC-H Q1 hash-aggregate input at SF100: 592 M rows x (2 x u8 keys + 5 x i64),
           sum x4, avg x3 (as sum+count states), count(*); 4 groups.
  agg_ssb  SSB Q4.1-shaped aggregate (configs[4]'s group-by): (d_year i32, c_nation u8) -> sum(profit), 35 groups.
  agg_q3   TPC-H Q3-shaped group-by (configs[3]'s): (l_orderkey i64, o_orderdate u16, o_shippriority u8) ->
           sum(revenue), 1 M groups (high cardinality: the L2-first table of agg_hc.cu).
  join     (configs[2]) TPC-H Q14 join at SF100: build part 20 M x (i64 key, u8 promo flag), probe 600 M lineitem
           rows x (i64 l_partkey, i64 l_extendedprice, i64 l_discount); every probe row matches one build row.
           At N > 1 THREE multi-GPU plans are measured: build side replicated (all-gather), the key-radix shuffle of
           both sides (peer scatter over NVLink), and the same with the probe side pipelined in chunks.
  scan     (configs[0] shape at SF100) l_shipdate < DATE '1994-01-01' -> l_quantity; row-range shards, no collective;
           `dictionary_vector`: the same predicate with l_shipdate as a DICTIONARY vector (generic interpreter).
  e2e_duckdb  (N = 1) TPC-H Q1 / Q14 / config 1 at SF1 INSIDE the unmodified reference through libb200_duckdb.so, next
           to the stock operators in the same connection.
  cpu_baseline  (N = 1) the reference on the box's usable cores on the first 60 M rows of every workload, with a
           bit-exact comparison of the GPU result on the same rows (`parity`).
A "step" is one pass of the operator over the whole input.  Every leg lists its K timed steps one by one (`ms_steps`);
`ms_per_step` / `value` are the K steps as ONE region, the sub-legs' rooflines use the median step.
`value` = rows/s with inputs resident in HBM;
`e2e` = the same through the C ABI from pinned HOST buffers (H2D of every input column and D2H of the result
inside the timed region, plus the cross-rank combine at N > 1).  At N > 1 every rank holds its own SF100-sized
shard (weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench_data as BD  # noqa: E402

SF100_LINEITEM = 600_037_902
Q1_ROWS = 591_855_000          # rows passing l_shipdate <= 1998-09-02 (98.64 %)
PART_ROWS = 20_000_000
AGG_BYTES_PER_ROW = 42         # SURVEY.md 8d / BASELINE.md section 4
JOIN_BYTES_PER_ROW = 73
SCAN_BYTES_PER_ROW = 14.2
SSB_BYTES_PER_ROW = 13         # i32 + u8 + i64
Q3_INPUT_BYTES_PER_ROW = 19    # i64 + u16 + u8 + i64
Q3_BYTES_PER_ROW = 51          # SURVEY.md 8d: inputs + one 32 B random state sector per row


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic():
    """DRAM bytes per row of the shipped kernels from the committed ncu --set full captures
    (profiles/r2_traffic.json, written by scripts/ncu_summary.py)."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def traffic_of(traffic, key, rows):
    t = traffic.get(key)
    if not t:
        return None, None
    return int(round(t["dram_bytes_per_row"] * rows)), t.get("source")


AGG_RESULT_COLUMNS = ("rf", "ls", "sum_qty", "sum_base_price", "sum_disc_price", "sum_charge", "avg_qty", "avg_price",
                      "avg_disc", "count_order")


def dump_agg_outputs(outdir, res):
    """The headline aggregate's result as outdir/agg_<column>.npy (float64), rows ordered by the group keys: the
    device hands the groups back in hash-table order, which may differ between builds.  float64 keeps only the top 53
    bits of a 128-bit sum, so each sum is also written exactly as agg_<column>_limbs.npy: its four 32-bit limbs in
    two's complement, least significant first."""
    os.makedirs(outdir, exist_ok=True)
    order = np.lexsort((res[1][0], res[0][0]))
    for name, (vals, _) in zip(AGG_RESULT_COLUMNS, res):
        vals = vals[order]
        if vals.dtype == object:
            words = [int(v) % (1 << 128) for v in vals]
            limbs = np.array([[(w >> (32 * i)) & 0xFFFFFFFF for i in range(4)] for w in words], dtype=np.float64)
            np.save(os.path.join(outdir, f"agg_{name}_limbs.npy"), limbs.reshape(len(words), 4))
            vals = np.array([float(v) for v in vals])
        np.save(os.path.join(outdir, f"agg_{name}.npy"), vals.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, device):
        self.device = device
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.device), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(float(f[0]))
                    self.max_mhz = float(f[1])
                    for nme, v in zip(names, f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(nme)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------- reference (CPU) arm
Q_AGG = ("SELECT rf, ls, sum(qty), sum(price), sum(disc_price), sum(charge), avg(qty), avg(price), avg(disc), "
         "count(*) FROM q1in GROUP BY rf, ls")
Q_JOIN = "SELECT count(*), sum(price), sum(disc), sum(promo) FROM li JOIN part ON li.partkey = part.partkey"
Q_SCAN = "SELECT sum(qty), count(*) FROM (SELECT qty FROM sc WHERE shipdate < 8766)"
Q_SSB = "SELECT year, nation, sum(profit) FROM ssb GROUP BY year, nation"
Q_Q3 = "SELECT okey, odate, prio, sum(revenue) FROM q3in GROUP BY okey, odate, prio"


class ReferenceRunner:
    """DuckDB's own operators (unmodified reference, oracle/_ref) on tables built from bench_data's formulas."""

    def __init__(self, threads):
        from oracle import duckdb_ref as R

        self.con = R.Connection(threads=threads)
        self.con.execute("SET preserve_insertion_order=false")
        self.threads = threads

    def timed(self, sql, warmup, steps, settings=(), budget_s=150.0):
        for s in settings:
            self.con.execute(s)
        t_begin = time.perf_counter()
        for _ in range(max(1, warmup)):
            self.con.execute(sql)
            if time.perf_counter() - t_begin > budget_s / 2:
                break
        ts = []
        for _ in range(max(1, steps)):
            t0 = time.perf_counter()
            self.con.execute(sql)
            ts.append(time.perf_counter() - t0)
            if time.perf_counter() - t_begin > budget_s:
                break
        return ts

    def close(self):
        self.con.close()


def run_reference_arm(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import duckdb_ref as R

    if not R.available():
        emit({"impl": "reference", "unavailable": "oracle/_ref/libduckdb_ref.so was not built"})
        return
    cores, core_info = BD.effective_cores()
    mem_gb = BD.mem_available_gb()
    # the same configuration as our arm when the host has the memory for it (SF100 Q1 input = 25 GB, probe side 14 GB)
    n = int(args.ref_rows) if args.ref_rows else (int(args.rows) if mem_gb >= 96 else 60_000_000)
    np_rows = int(args.ref_rows) if args.ref_rows else (int(args.probe_rows) if mem_gb >= 96 else 60_000_000)
    nb = max(1000, int(args.build_rows * np_rows / args.probe_rows))
    K, W = max(1, args.steps), max(1, args.warmup)
    ref = ReferenceRunner(cores)
    t0 = time.perf_counter()
    ref.con.execute(BD.q1_table_sql("q1in", n))
    t_create = time.perf_counter() - t0
    ts_stock = ref.timed(Q_AGG, W, K, ["RESET perfect_ht_threshold"], budget_s=120)
    ts_hash = ref.timed(Q_AGG, min(W, 2), min(K, 5), ["SET perfect_ht_threshold=0"], budget_s=60)
    ref.con.execute("RESET perfect_ht_threshold")
    stock, hashed = n / float(np.mean(ts_stock)), n / float(np.mean(ts_hash))
    agg = max(stock, hashed)
    ts = ts_stock if stock >= hashed else ts_hash
    ref.con.execute("DROP TABLE q1in")
    line = {
        "impl": "reference", "metric": "agg_input_rows_per_s", "value": agg, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": len(ts), "warmup": W, "ms_per_step": 1000.0 * n / agg, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "TPC-H Q1 hash-aggregate, SF100 lineitem (BASELINE configs[1])", "rows": n,
                   "full_size": n == args.rows, "table_build_s": t_create,
                   "plan": "faster of DuckDB's stock plan (PERFECT_HASH_GROUP_BY) and HASH_GROUP_BY (perfect_ht_threshold=0)"},
        "cpu_baseline": {"value": agg, "unit": "rows/s", "cores": cores, "kind": "reference",
                         "core_info": core_info, "host_mem_available_gb": mem_gb,
                         "sample": f"{n} rows of the SF100 Q1 input per step ({'the full configuration' if n == args.rows else 'bounded by host memory'}), "
                                   f"SET threads={cores}",
                         "agg_hash_group_by_rows_per_s": hashed, "agg_stock_plan_rows_per_s": stock},
        "e2e": {"value": agg, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    try:
        ref.con.execute(BD.probe_table_sql("li", np_rows, nb))
        ref.con.execute(BD.part_table_sql("part", nb))
        tj = ref.timed(Q_JOIN, 1, min(K, 3), ["SET disabled_optimizers='join_filter_pushdown'"], budget_s=90)
        ref.con.execute("RESET disabled_optimizers")
        join = np_rows / float(np.mean(tj))
        line["join_probe"] = {"value": join, "unit": "rows/s", "probe_rows": np_rows, "build_rows": nb, "steps": len(tj),
                              "e2e": {"value": join, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        ref.con.execute("DROP TABLE li")
        ref.con.execute(BD.scan_table_sql("sc", np_rows))
        tsn = ref.timed(Q_SCAN, 1, min(K, 3), budget_s=60)
        line["scan"] = {"value": np_rows / float(np.mean(tsn)), "unit": "rows/s", "rows": np_rows}
    except Exception as ex:  # the secondary legs must not take the headline down
        line["join_probe"] = line.get("join_probe", {"error": f"{type(ex).__name__}: {ex}"})
    ref.close()
    emit(line)


def cpu_baseline_leg(args, rank0_checks):
    """Bounded sample of every workload on the host cores (rank 0, N = 1), with the reference's per-group results
    handed to `rank0_checks` so that the GPU results on the same rows can be compared bit for bit."""
    from oracle import duckdb_ref as R

    if not R.available():
        return {"value": None, "unit": "rows/s", "cores": 0, "kind": "reference",
                "sample": "oracle/_ref/libduckdb_ref.so not present"}
    cores, core_info = BD.effective_cores()
    n = int(args.cpu_rows)
    nb = max(1000, int(args.build_rows * n / args.probe_rows))
    ref = ReferenceRunner(cores)
    out = {"unit": "rows/s", "cores": cores, "kind": "reference", "core_info": core_info,
           "sample": f"first {n} rows of every workload (1 warm-up + 3 runs, mean), SET threads={cores}"}
    ref.con.execute(BD.q1_table_sql("q1in", n))
    stock = n / float(np.mean(ref.timed(Q_AGG, 1, 3, ["RESET perfect_ht_threshold"])))
    hashed = n / float(np.mean(ref.timed(Q_AGG, 1, 3, ["SET perfect_ht_threshold=0"])))
    ref.con.execute("RESET perfect_ht_threshold")
    out.update({"value": max(stock, hashed), "agg_stock_plan_rows_per_s": stock, "agg_hash_group_by_rows_per_s": hashed})
    rows = ref.con.fetchall(Q_AGG)
    out["parity"] = {"agg_q1": rank0_checks["q1"](n, rows)}
    ref.con.execute("DROP TABLE q1in")
    ref.con.execute(BD.ssb_table_sql("ssb", n))
    out["agg_ssb_rows_per_s"] = n / float(np.mean(ref.timed(Q_SSB, 1, 3)))
    out["parity"]["agg_ssb"] = rank0_checks["ssb"](n, ref.con.fetchall(Q_SSB))
    ref.con.execute("DROP TABLE ssb")
    nq3 = min(n, int(args.q3_rows))
    ref.con.execute(BD.q3_table_sql("q3in", nq3, int(args.q3_groups)))
    out["agg_q3_rows_per_s"] = nq3 / float(np.mean(ref.timed(Q_Q3, 1, 3)))
    out["parity"]["agg_q3"] = rank0_checks["q3"](nq3, ref.con.fetchall(
        "SELECT count(*), sum(s), sum(okey * (s % 1000003)) FROM (" + Q_Q3.replace("sum(revenue)", "sum(revenue) AS s") + ")"))
    ref.con.execute("DROP TABLE q3in")
    ref.con.execute(BD.probe_table_sql("li", n, nb))
    ref.con.execute(BD.part_table_sql("part", nb))
    tj = ref.timed(Q_JOIN, 1, 3, ["SET disabled_optimizers='join_filter_pushdown'"])
    ref.con.execute("RESET disabled_optimizers")
    out["join_probe_rows_per_s"] = n / float(np.mean(tj))
    out["parity"]["join"] = rank0_checks["join"](n, nb, ref.con.fetchall(Q_JOIN))
    ref.con.execute("DROP TABLE li")
    ref.con.execute(BD.scan_table_sql("sc", n))
    out["scan_rows_per_s"] = n / float(np.mean(ref.timed(Q_SCAN, 1, 3)))
    out["parity"]["scan"] = rank0_checks["scan"](n, ref.con.fetchall(Q_SCAN))
    ref.close()
    return out


# --------------------------------------------------------------------------- our arm
def main():
    # only the JSON line may reach stdout: libraries (NCCL prints its version banner) get stderr instead
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--rows", type=int, default=Q1_ROWS, help="aggregate input rows per GPU")
    ap.add_argument("--probe-rows", type=int, default=SF100_LINEITEM)
    ap.add_argument("--build-rows", type=int, default=PART_ROWS)
    ap.add_argument("--ssb-rows", type=int, default=SF100_LINEITEM)
    ap.add_argument("--q3-rows", type=int, default=256_000_000)
    ap.add_argument("--q3-groups", type=int, default=1_000_000)
    ap.add_argument("--ref-rows", type=int, default=0, help="reference arm: rows per step (0 = the full configuration "
                                                            "when the host has the memory, else 60 M)")
    ap.add_argument("--cpu-rows", type=int, default=60_000_000, help="rows of the bounded cpu_baseline sample")
    ap.add_argument("--join-plan", default="both", choices=["both", "broadcast", "shuffle", "shuffle_pipelined"],
                    help="multi-GPU join plan(s) to measure")
    ap.add_argument("--duckdb-sf", type=float, default=1.0, help="TPC-H scale factor of the e2e_duckdb leg")
    ap.add_argument("--skip", default="", help="comma list of legs to skip: ssb,q3,join,scan,e2e,duckdb,cpu")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline aggregate's result of the last timed step "
                                                          "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args, emit)
        return
    skip = set(x for x in args.skip.split(",") if x)

    import torch
    import torch.distributed as dist

    from duckdb_b200 import capi
    from duckdb_b200 import operators as ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        # measured on 2 x B200: changing the persisting-L2 carve-out around every probe (b200_l2_pin/unpin) while
        # NCCL is active costs ~0.4 s per call (and the carve-out is opt-in since round 2 anyway)
        os.environ["B200_NO_L2_PIN"] = "1"
    ctx = ops.Context(local_rank, torch.cuda.current_stream().cuda_stream)
    peak, peak_src = load_peaks()
    traffic = load_traffic()
    K, W = args.steps, max(3, args.warmup)
    gen = BD.Gen(torch, dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def sum_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.int64, device=dev)
            dist.all_reduce(t)
            return int(t.item())
        return int(x)

    def all_ranks_ok(ok):
        """True only when every rank says so (so that no rank waits in a barrier for one that gave up)."""
        if world > 1:
            t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return bool(t.item())
        return bool(ok)

    def timed_steps(step, warmup=W, steps=K):
        """W untimed + K timed steps, barrier + synchronize on both sides, device time, max over ranks -> ms/step"""
        for _ in range(warmup):
            step()
        if True:  # (also with warmup=0: the headline does its own warm-up loop)
            # one more untimed step AFTER a device-wide synchronise: on this pool the first step that follows a
            # torch.cuda.synchronize() sometimes stalls once for ~0.1-0.7 s (seen in the scan leg only, per-step times in
            # `ms_steps` of profiles/r2_bench_n1.json: [101.5, 1.63, 1.58, 1.59, 1.57]); it is not part of any step's work
            barrier()
            step()
        timed_steps.stalled = None
        for attempt in range(2):
            barrier()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            ev[0].record()
            for i in range(steps):
                step()
                ev[i + 1].record()
            barrier()
            # the K steps as ONE region (the contract) plus every step on its own (a one-off stall shows up here)
            per_step = [round(ev[i].elapsed_time(ev[i + 1]), 4) for i in range(steps)]
            region = ev[0].elapsed_time(ev[steps])
            # a single step more than 2 x the median step is a stall of the box, not of the operator (100 ms .. 0.7 s
            # have been seen on 1.6 .. 10 ms steps): like the driver does for a throttled run, the K-step region is
            # measured ONCE more and the discarded per-step times are reported next to the kept ones.  Every rank must
            # take the same decision (the steps contain collectives).
            stalled = steps >= 3 and max(per_step) > 2.0 * float(np.median(per_step))
            if world > 1:
                flag = torch.tensor([1 if stalled else 0], dtype=torch.int64, device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
                stalled = bool(flag.item())
            if attempt == 0 and stalled:
                timed_steps.stalled = per_step
                continue
            break
        timed_steps.last = per_step
        return max_over_ranks(region) / steps

    def roofline(bytes_per_row, rows, ms, kernel, traffic_key=None, note=None):
        gbs = bytes_per_row * rows / (ms / 1e3) / 1e9
        tr, src = traffic_of(traffic, traffic_key, rows) if traffic_key else (None, None)
        r = {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": tr,
             "kernel": kernel, "ms": ms, "peak_source": peak_src, "bytes_per_row": bytes_per_row,
             "ms_stat": "headline: mean of the K sink calls; other legs: MEDIAN of the K timed steps / sink calls (every "
                        "step is in ms_steps; the shared boxes of this pool show one-off stalls of 8-700 ms in single steps)"}
        if src:
            r["traffic_source"] = src
        if note:
            r["note"] = note
        return r

    def wrap(cols, types, n):
        return ops.Batch.wrap(ctx, [(t.data_ptr(), ty) for t, ty in zip(cols, types)], n, keepalive=cols)

    checks = {}

    # ----------------------------------------------------------------- aggregate Q1 (headline)
    n = args.rows
    q1 = gen.q1(n, rank * n)
    agg_cols = [q1[k] for k in ("rf", "ls", "qty", "price", "disc_price", "charge", "disc")]
    agg_types = [capi.UINT8, capi.UINT8] + [capi.INT64] * 5
    # aggregate inputs: 0 qty, 1 price, 2 disc_price, 3 charge, 4 disc  (sum(qty)/avg(qty) etc. share their input)
    agg_desc = [(capi.AGG_SUM, capi.INT64, 0), (capi.AGG_SUM, capi.INT64, 1), (capi.AGG_SUM, capi.INT64, 2),
                (capi.AGG_SUM, capi.INT64, 3), (capi.AGG_AVG, capi.INT64, 0), (capi.AGG_AVG, capi.INT64, 1),
                (capi.AGG_AVG, capi.INT64, 4), (capi.AGG_COUNT_STAR, capi.INT64, -1)]
    agg_in = [2, 3, 4, 5, 6]
    resident = wrap(agg_cols, agg_types, n)
    sink_events = []

    def finish_agg(a, key_types, desc):
        """cross-rank combine (N > 1: ONE all-gather of packed partial states + ONE merge kernel) + finalize + download"""
        if world > 1:
            from duckdb_b200.distributed import allgather_agg_states

            f = ops.HashAggregate(ctx, key_types, desc)
            allgather_agg_states(ctx, a, f)
            res = f.finalize().download_all()
            f.close()
        else:
            res = a.finalize().download_all()
        a.close()
        return res

    def agg_step(batches=None, timed=True):
        a = ops.HashAggregate(ctx, [capi.UINT8, capi.UINT8], agg_desc)
        for b in (batches or [resident]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a.sink(b, [0, 1], agg_in)
            e1.record()
            if timed:
                sink_events.append((e0, e1))
        agg_step.res = finish_agg(a, [capi.UINT8, capi.UINT8], agg_desc)

    sampler = ClockSampler(local_rank)
    for _ in range(W):
        agg_step(timed=False)
    sampler.start()
    stats0 = ctx.stats()
    agg_ms = timed_steps(agg_step, warmup=0)
    agg_steps_ms = list(timed_steps.last)
    agg_stalled = timed_steps.stalled
    clocks = sampler.stop()
    res = agg_step.res
    # K timed steps + the settling step (+ K more if the region was measured a second time after a stall)
    launches = (ctx.stats()["launches"] - stats0["launches"]) // (K + 1 + (K if agg_stalled else 0))
    sink_ms = float(np.mean([a.elapsed_time(b) for a, b in sink_events[-K:]]))
    agg_value = world * n / (agg_ms / 1e3)
    # sanity: the result must be the right one (count(*) sums to the input rows; sums match torch's)
    cnt_total = int(res[9][0].sum())
    assert cnt_total == n * world, (cnt_total, n * world)
    assert sum(int(x) for x in res[2][0]) == sum_over_ranks(int(q1["qty"].sum().item())), "sum(qty) mismatch"
    if args.dump_outputs and rank == 0:
        dump_agg_outputs(args.dump_outputs, res)

    def groups_of(res, nkeys):
        return {tuple(int(res[j][0][g]) for j in range(nkeys)): [res[nkeys + a][0][g] for a in range(len(res) - nkeys)]
                for g in range(len(res[0][0]))}

    def check_q1(m, ref_rows):
        """GPU aggregate of the first m rows vs the reference's answer on the same rows: sums / counts bit-exact,
        averages within 1e-9 relative (BASELINE.json north_star)"""
        a = ops.HashAggregate(ctx, [capi.UINT8, capi.UINT8], agg_desc)
        a.sink(wrap(agg_cols, agg_types, m), [0, 1], agg_in)
        got = groups_of(a.finalize().download_all(), 2)
        a.close()
        if len(got) != len(ref_rows):
            return f"MISMATCH: {len(got)} groups vs {len(ref_rows)}"
        for r in ref_rows:
            g = got[(int(r[0]), int(r[1]))]
            if [int(x) for x in g[:4]] != [int(x) for x in r[2:6]] or int(g[7]) != int(r[9]):
                return f"MISMATCH in group {r[0]},{r[1]}"
            for x, y in zip(g[4:7], r[6:9]):
                if abs(float(x) - float(y)) > 1e-9 * abs(float(y)):
                    return f"MISMATCH avg in group {r[0]},{r[1]}"
        return f"bit-exact on {m} rows ({len(got)} groups: 4 hugeint sums + count, 3 avgs within 1e-9)"

    checks["q1"] = check_q1
    tr, trsrc = traffic_of(traffic, "agg_fastreg", n)
    line = {
        "metric": "agg_input_rows_per_s", "value": agg_value, "unit": "rows/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": agg_ms, "ms_steps": agg_steps_ms, "ms_steps_discarded": agg_stalled, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": "TPC-H Q1 hash-aggregate, SF100 lineitem (BASELINE configs[1])",
                   "rows_per_gpu": n, "row_bytes": AGG_BYTES_PER_ROW, "groups": 4,
                   "aggregates": "sum x4 (hugeint), avg x3, count(*)",
                   "l2": "inputs (24.9 GB) larger than L2", "parallelism": f"shard{world}",
                   "combine": "none (N = 1)" if world == 1 else "all-gather of packed partial states + one merge kernel, "
                                                                "inside every timed step"},
        "roofline": roofline(AGG_BYTES_PER_ROW, n, sink_ms,
                             "agg_fastreg_kernel<5,4,224,1> (b200_agg_sink, incl. the 256 K-row adaptation probe)",
                             "agg_fastreg"),
        "gpu_launches": int(launches), "clocks": clocks,
    }

    # ----------------------------------------------------------------- e2e aggregate (host buffers)
    host = None
    if "e2e" not in skip:
        # 24.9 GB of pinned host memory per rank: if the box cannot give that to every rank, report the e2e leg as
        # unavailable instead of losing the whole line
        try:
            host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in agg_cols]
            for h, t in zip(host, agg_cols):
                h.copy_(t)
            torch.cuda.synchronize()
        except Exception as ex:
            sys.stderr.write(f"[bench] rank {rank}: pinned host buffers for the e2e leg failed: {ex!r}\n")
            host = None
        if not all_ranks_ok(host is not None):
            host = None
            line["e2e"] = {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                           "error": "pinned host staging buffers could not be allocated on every rank"}
    if host is not None:
        host_np = [h.numpy() for h in host]
        chunk = 1 << 26

        def e2e_step():
            a = ops.HashAggregate(ctx, [capi.UINT8, capi.UINT8], agg_desc)
            for lo in range(0, n, chunk):
                hi = min(n, lo + chunk)
                b = ops.Batch.upload(ctx, [ops.Vector.flat(c[lo:hi]) for c in host_np], hi - lo)
                a.sink(b, [0, 1], agg_in)
                b.free()
            return finish_agg(a, [capi.UINT8, capi.UINT8], agg_desc)

        e2e_step()
        s0 = ctx.stats()
        barrier()
        w0 = time.perf_counter()
        ksteps = max(1, min(K, 3))
        for _ in range(ksteps):
            r2 = e2e_step()
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - w0) / ksteps
        s1 = ctx.stats()
        assert int(r2[9][0].sum()) == n * world
        line["e2e"] = {"value": world * n / e2e_s, "unit": "rows/s",
                       "h2d_bytes_per_step": int((s1["h2d_bytes"] - s0["h2d_bytes"]) // ksteps),
                       "d2h_bytes_per_step": int((s1["d2h_bytes"] - s0["d2h_bytes"]) // ksteps),
                       "ms_per_step": e2e_s * 1e3, "h2d_gbs_per_gpu": AGG_BYTES_PER_ROW * n / e2e_s / 1e9,
                       "note": "pinned host columns -> b200_batch_upload (64 Mi-row morsels) -> sink -> "
                               + ("cross-rank combine -> " if world > 1 else "") + "finalize -> D2H of the result"}
        del host, host_np

    # ----------------------------------------------------------------- SSB Q4.1-shaped aggregate (35 groups)
    def guarded(name, fn):
        try:
            fn()
        except Exception as ex:  # a secondary leg must never take the headline number down with it
            import traceback

            traceback.print_exc()
            line[name] = {"error": f"{type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()

    def leg_ssb():
        ns = args.ssb_rows
        d = gen.ssb(ns, rank * ns)
        cols, types = [d["year"], d["nation"], d["profit"]], [capi.INT32, capi.UINT8, capi.INT64]
        desc = [(capi.AGG_SUM, capi.INT64, 0)]
        batch = wrap(cols, types, ns)
        ev = []

        def step():
            a = ops.HashAggregate(ctx, types[:2], desc)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a.sink(batch, [0, 1], [2])
            e1.record()
            ev.append((e0, e1))
            step.res = finish_agg(a, types[:2], desc)

        ms = timed_steps(step)
        steps_ms = list(timed_steps.last)
        stalled_ms = timed_steps.stalled
        sink = float(np.median([a.elapsed_time(b) for a, b in ev[-K:]]))   # median: a one-off stall is not the kernel
        got = groups_of(step.res, 2)
        assert len(got) == 35, len(got)
        assert sum(int(v[0]) for v in got.values()) == sum_over_ranks(int(d["profit"].sum().item())), "sum(profit) mismatch"

        def check(m, ref_rows):
            a = ops.HashAggregate(ctx, types[:2], desc)
            a.sink(wrap(cols, types, m), [0, 1], [2])
            g = groups_of(a.finalize().download_all(), 2)
            a.close()
            ok = len(g) == len(ref_rows) and all(int(g[(int(r[0]), int(r[1]))][0]) == int(r[2]) for r in ref_rows)
            return f"bit-exact on {m} rows ({len(g)} groups)" if ok else "MISMATCH"

        checks["ssb"] = check
        line["agg_ssb"] = {
            "metric": "agg_input_rows_per_s", "value": world * ns / (ms / 1e3), "unit": "rows/s", "ms_per_step": ms,
            "ms_steps": steps_ms, "ms_steps_discarded": stalled_ms,
            "config": {"workload": "SSB Q4.1-shaped aggregate (BASELINE configs[4]'s group-by): GROUP BY d_year, c_nation "
                                   "SUM(lo_revenue - lo_supplycost); every row of an SF100-sized shard (stress)",
                       "rows_per_gpu": ns, "row_bytes": SSB_BYTES_PER_ROW, "groups": 35},
            "roofline": roofline(SSB_BYTES_PER_ROW, ns, sink, "agg_priv_kernel<1,0> (thread-private shared-memory accumulators)",
                                 "agg_priv1")}
        checks["_keep_ssb"] = (cols, batch)

    if "ssb" not in skip:
        guarded("agg_ssb", leg_ssb)

    # ----------------------------------------------------------------- TPC-H Q3-shaped group-by (1 M groups)
    def leg_q3():
        nq, groups = args.q3_rows, args.q3_groups
        d = gen.q3(nq, groups, rank * nq)
        cols = [d["okey"], d["odate"], d["prio"], d["revenue"]]
        types = [capi.INT64, capi.UINT16, capi.UINT8, capi.INT64]
        desc = [(capi.AGG_SUM, capi.INT64, 0)]
        batch = wrap(cols, types, nq)
        ev = []

        def local_agg(b):
            a = ops.HashAggregate(ctx, types[:3], desc)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a.sink(b, [0, 1, 2], [3])
            e1.record()
            ev.append((e0, e1))
            out = a.finalize()
            a.close()
            return out

        def step():
            if world > 1:
                # high-cardinality multi-GPU plan (SURVEY.md 8e): shuffle the ROWS by key radix, aggregate locally,
                # no merge - every group lives on exactly one GPU
                from duckdb_b200.distributed import shuffle_batch

                mine, keep = shuffle_batch(ctx, batch, [0, 1, 2])
                out = local_agg(mine)
                mine.free()
                del keep
            else:
                out = local_agg(batch)
            step.groups = out.nrows
            step.out = out

        ms = timed_steps(step)
        steps_ms = list(timed_steps.last)
        stalled_ms = timed_steps.stalled
        sink = float(np.median([a.elapsed_time(b) for a, b in ev[-K:]]))   # median: a one-off stall is not the kernel
        tot_groups = sum_over_ranks(step.groups)
        res = step.out.download_all()
        tot_sum = sum_over_ranks(sum(int(x) for x in res[3][0]))
        assert tot_sum == sum_over_ranks(int(d["revenue"].sum().item())), "sum(revenue) mismatch"
        if world == 1:
            assert tot_groups == int(torch.unique(d["okey"]).numel()), "group count mismatch"

        def check(m, ref_rows):
            a = ops.HashAggregate(ctx, types[:3], desc)
            a.sink(wrap(cols, types, m), [0, 1, 2], [3])
            r = a.finalize().download_all()
            a.close()
            ok = np.array([int(x) for x in r[0][0]], dtype=object)
            s = np.array([int(x) for x in r[3][0]], dtype=object)
            mine = (len(ok), int(s.sum()), int((ok * (s % 1000003)).sum()))
            want = tuple(int(x) for x in ref_rows[0])
            return (f"bit-exact on {m} rows ({mine[0]} groups: group count, total and a key-weighted checksum of the "
                    f"per-group sums)") if mine == want else f"MISMATCH {mine} vs {want}"

        checks["q3"] = check
        line["agg_q3"] = {
            "metric": "agg_input_rows_per_s", "value": world * nq / (ms / 1e3), "unit": "rows/s", "ms_per_step": ms,
            "ms_steps": steps_ms, "ms_steps_discarded": stalled_ms,
            "groups": tot_groups,
            "config": {"workload": "TPC-H Q3-shaped group-by (BASELINE configs[3]'s): GROUP BY l_orderkey, o_orderdate, "
                                   "o_shippriority SUM(revenue); stress: every input row, not only the join survivors",
                       "rows_per_gpu": nq, "input_row_bytes": Q3_INPUT_BYTES_PER_ROW, "row_bytes": Q3_BYTES_PER_ROW,
                       "groups": groups,
                       "plan": "local" if world == 1 else "rows shuffled by key radix (all-to-all), local aggregate, no merge"},
            "roofline": roofline(Q3_BYTES_PER_ROW, nq, sink, "agg_hc_direct_kernel<2,1> (L2-first structure-of-arrays table; "
                                 "sink incl. the adaptation probe, chunking and table growth)", "agg_hc",
                                 note="SURVEY 8d's 51 B/row: 19 B of inputs + one 32 B random state sector per row; the table "
                                      "(1 M groups = 48 MB) stays in L2, so DRAM traffic is the 19 B/row of inputs")}
        checks["_keep_q3"] = (cols, batch)

    if "q3" not in skip:
        guarded("agg_q3", leg_q3)
    del resident
    torch.cuda.empty_cache()

    # ----------------------------------------------------------------- join probe (configs[2])
    def leg_join():
        from duckdb_b200.distributed import allgather_columns, shuffle_batch

        nb, npb = args.build_rows, args.probe_rows
        nb_total = nb * world                                # weak scaling: SF100 x world
        part = gen.part(nb, 1 + rank * nb)                   # this rank's shard of part: a contiguous key range
        probe = gen.probe(npb, nb_total, rank * npb)         # probe keys reference the whole key space
        bk, bp = part["partkey"], part["promo"]
        pk, pprice, pdisc = probe["partkey"], probe["price"], probe["disc"]
        bbatch = wrap([bk, bp], [capi.INT64, capi.UINT8], nb)
        pbatch = wrap([pk, pprice, pdisc], [capi.INT64] * 3, npb)

        def run_plan(plan):
            j = ops.HashJoin(ctx, capi.JOIN_INNER, [capi.INT64], [capi.UINT8])
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            keep = None
            if plan.startswith("shuffle"):
                bmine, keep = shuffle_batch(ctx, bbatch, [0])     # build side partitioned by key radix
                j.sink(bmine, [0], [1])
            elif plan == "broadcast":
                ball = allgather_columns([bk, bp])                 # every rank builds the whole (small) build side
                keep = ball
                j.sink(wrap(ball, [capi.INT64, capi.UINT8], nb_total), [0], [1])
            else:
                j.sink(bbatch, [0], [1])
            j.finalize()
            b1.record()
            torch.cuda.synchronize()
            build_ms = max_over_ranks(b0.elapsed_time(b1))

            from duckdb_b200.distributed import _DevArray

            def checksum(o):
                """sum of the joined price column (every probe row matches exactly one build row: it must add up)"""
                nout = o.nrows
                inf = o.column_info(0)
                return int(torch.as_tensor(_DevArray(inf.data, nout, "<i8"), device=dev).sum().item()) if nout else 0

            pipe = None
            if plan in ("shuffle", "shuffle_pipelined") and os.environ.get("B200_SHUFFLE", "peer") == "peer" and \
                    plan == "shuffle_pipelined":
                from duckdb_b200.distributed import PipelinedShuffleProbe

                pipe = PipelinedShuffleProbe(ctx, j, [capi.INT64] * 3, npb, nchunks=4)

            def probe_step():
                probe_step.sum = 0
                if pipe is not None:
                    def consume(o, c):
                        if probe_step.check:
                            probe_step.sum += checksum(o)
                        o.free()

                    probe_step.cnt = pipe.probe(pbatch, [0], [1, 2], consume)
                    return
                if plan.startswith("shuffle"):
                    pmine, pkeep = shuffle_batch(ctx, pbatch, [0])  # probe side follows the same radix partitioning
                    o, c = j.execute(pmine, [0], [1, 2])
                    pmine.free()
                    del pkeep
                else:
                    o, c = j.execute(pbatch, [0], [1, 2])
                probe_step.cnt = c
                if probe_step.check:
                    probe_step.sum = checksum(o)
                o.free()

            probe_step.check = False
            ms = timed_steps(probe_step)
            steps_ms = list(timed_steps.last)
            stalled_ms = timed_steps.stalled
            probe_step.check = True
            probe_step()   # one more, untimed, with the checksum of the joined column
            assert sum_over_ranks(probe_step.cnt) == npb * world, (probe_step.cnt, npb)
            assert sum_over_ranks(probe_step.sum) == sum_over_ranks(int(pprice.sum().item())), "joined sum(price) mismatch"
            res = {"ms": ms, "ms_steps": steps_ms, "ms_steps_discarded": stalled_ms, "build_ms": build_ms, "value": world * npb / (ms / 1e3), "join": j,
                   "out": None}
            del keep
            return res

        plans = ["local"] if world == 1 else (["broadcast", "shuffle", "shuffle_pipelined"] if args.join_plan == "both"
                                              else [args.join_plan])
        results = {}
        for p in plans:
            results[p] = run_plan(p)
        main_plan = plans[0]
        r = results[main_plan]
        dense_note = ("achieved uses SURVEY 8d's 73 B/row; with the dense (perfect-hash) table the 32 B random sector is a "
                      "4 B L2-resident entry, i.e. 45 B/row actually move")
        plan_text = {"local": "local build/probe",
                     "broadcast": "build side replicated on every GPU (NCCL all-gather, inside build_ms), probe side in "
                                  "place: no exchange on the probe pipeline",
                     "shuffle": "key-radix shuffle of both sides (one fused partition + NVLink peer-scatter kernel per "
                                "source GPU), then local build/probe; the probe-side shuffle is inside every timed step",
                     "shuffle_pipelined": "same, the probe side in 4 chunks: chunk c+1 crosses NVLink on a second "
                                          "stream while chunk c is probed"}
        line["join_probe"] = {
            "metric": "join_probe_rows_per_s", "value": r["value"], "unit": "rows/s", "ms_per_step": r["ms"],
            "ms_steps": r["ms_steps"], "ms_steps_discarded": r["ms_steps_discarded"],
            "n_gpus": world, "plan": plan_text[main_plan],
            "config": {"workload": "TPC-H Q14 lineitem x part hash join, SF100 per GPU (BASELINE configs[2], 3b stress: "
                                   "all 600 M probe rows)", "build_rows_per_gpu": nb,
                       "hash_table_rows_per_gpu": nb_total if main_plan == "broadcast" else nb, "probe_rows_per_gpu": npb,
                       "row_bytes": JOIN_BYTES_PER_ROW, "l2": "probe inputs (14.4 GB) larger than L2"},
            "build_ms": r["build_ms"], "build_rows_per_s": world * nb / (r["build_ms"] / 1e3),
            "roofline": roofline(JOIN_BYTES_PER_ROW, npb, float(np.median(r["ms_steps"])), "join_probe_lean2_kernel<2,8,dense>", "join_dense",
                                 note=dense_note)}
        for p in plans[1:]:
            q = results[p]
            line["join_probe_" + p] = {
                "metric": "join_probe_rows_per_s", "value": q["value"], "unit": "rows/s", "ms_per_step": q["ms"],
                "ms_steps": q["ms_steps"], "ms_steps_discarded": q["ms_steps_discarded"],
                "n_gpus": world, "plan": plan_text[p], "build_ms": q["build_ms"],
                "nvlink_bytes_per_step_per_gpu": int(npb * 24 * (world - 1) / world),
                "roofline": roofline(JOIN_BYTES_PER_ROW, npb, q["ms"], "part_count + part_move_staged + all-to-all + "
                                                                         "join_probe_tile_kernel", None)}

        def check(m, nbs, ref_rows):
            """first m probe rows against a build side of nbs keys (the reference's bounded sample)"""
            pr = gen.probe(m, nbs, 0)
            pt = gen.part(nbs, 1)
            jj = ops.HashJoin(ctx, capi.JOIN_INNER, [capi.INT64], [capi.UINT8])
            jj.sink(wrap([pt["partkey"], pt["promo"]], [capi.INT64, capi.UINT8], nbs), [0], [1])
            jj.finalize()
            o, c = jj.execute(wrap([pr["partkey"], pr["price"], pr["disc"]], [capi.INT64] * 3, m), [0], [1, 2])
            from duckdb_b200.distributed import _DevArray
            inf = [o.column_info(i) for i in range(3)]
            got = (c, int(torch.as_tensor(_DevArray(inf[0].data, c, "<i8"), device=dev).sum().item()),
                   int(torch.as_tensor(_DevArray(inf[1].data, c, "<i8"), device=dev).sum().item()),
                   int(torch.as_tensor(_DevArray(inf[2].data, c, "|u1"), device=dev).sum(dtype=torch.int64).item()))
            o.free()
            jj.close()
            want = tuple(int(x) for x in ref_rows[0])
            return f"bit-exact on {m} probe rows (row count, sum(price), sum(disc), sum(promo))" if got == want else \
                f"MISMATCH {got} vs {want}"

        checks["join"] = check
        if "e2e" not in skip and world == 1:
            j = r["join"]
            hk = torch.empty(npb, dtype=torch.int64, pin_memory=True)
            hp = torch.empty(npb, dtype=torch.int64, pin_memory=True)
            hd = torch.empty(npb, dtype=torch.int64, pin_memory=True)
            hk.copy_(pk), hp.copy_(pprice), hd.copy_(pdisc)
            torch.cuda.synchronize()
            hnp = [hk.numpy(), hp.numpy(), hd.numpy()]
            chunk = 1 << 26
            # pinned result buffers (price, discount, promo) for the D2H leg
            o_pin = [torch.empty(chunk, dtype=torch.int64, pin_memory=True), torch.empty(chunk, dtype=torch.int64, pin_memory=True),
                     torch.empty(chunk, dtype=torch.uint8, pin_memory=True)]

            def join_e2e():
                tot = 0
                for lo in range(0, npb, chunk):
                    hi = min(npb, lo + chunk)
                    b = ops.Batch.upload(ctx, [ops.Vector.flat(c[lo:hi]) for c in hnp], hi - lo)
                    o, c = j.execute(b, [0], [1, 2])
                    for ci in range(3):   # D2H of the joined columns
                        o.download_into(ci, o_pin[ci].data_ptr())
                    tot += c
                    o.free()
                    b.free()
                return tot

            join_e2e()
            s0 = ctx.stats()
            barrier()
            w0 = time.perf_counter()
            tot = join_e2e()
            barrier()
            dt = time.perf_counter() - w0
            s1 = ctx.stats()
            assert tot == npb
            line["join_probe"]["e2e"] = {"value": npb / dt, "unit": "rows/s",
                                         "h2d_bytes_per_step": int(s1["h2d_bytes"] - s0["h2d_bytes"]),
                                         "d2h_bytes_per_step": int(s1["d2h_bytes"] - s0["d2h_bytes"]), "ms_per_step": dt * 1e3}
            del hk, hp, hd, hnp
        for q in results.values():
            q["join"].close()
        torch.cuda.empty_cache()

    if "join" not in skip:
        guarded("join_probe", leg_join)

    # ----------------------------------------------------------------- filter scan (configs[0] shape at SF100)
    def leg_scan():
        ns = args.probe_rows
        d = gen.scan(ns, rank * ns)
        shipdate, quantity = d["shipdate"], d["qty"]
        sb = wrap([shipdate, quantity], [capi.INT32, capi.INT64], ns)
        e = ops.Expr()
        root = e.cmp(capi.EXPR_LT, e.col(0, capi.INT32), e.const(8766, capi.INT32))  # DATE '1994-01-01'
        fp = ops.FilterProject(ctx, e, root, [e.col(1, capi.INT64)])

        def step():
            o, c, _, _ = fp.execute(sb)
            step.c = c
            step.sum = None
            if step.keep:
                step.o = o
            else:
                o.free()

        step.keep = False
        if os.environ.get("BENCH_SCAN_DIAG"):
            def log(msg):
                sys.stderr.write(msg + "\n")
                sys.stderr.flush()

            free_b, total_b = torch.cuda.mem_get_info(dev)
            log(f"[scan diag] free {free_b / 1e9:.1f} GB of {total_b / 1e9:.1f} GB, torch reserved "
                f"{torch.cuda.memory_reserved(dev) / 1e9:.1f} GB")
            for i in range(6):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                step()
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                x = shipdate.clone()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                del x
                log(f"[scan diag] step {i}: {1e3 * (t1 - t0):.2f} ms wall, clone of 2.4 GB {1e3 * (t2 - t1):.2f} ms")
        scan_ms = timed_steps(step)
        scan_steps = list(timed_steps.last)
        scan_stalled = timed_steps.stalled
        c = step.c
        assert c == int((shipdate < 8766).sum().item()), "scan count mismatch"
        scan_bytes = ns * 12 + c * 8
        line["scan"] = {"metric": "scan_filter_rows_per_s", "value": world * ns / (scan_ms / 1e3), "unit": "rows/s",
                        "ms_per_step": scan_ms, "ms_steps": scan_steps, "ms_steps_discarded": scan_stalled, "selectivity": c / ns, "n_gpus": world,
                        "config": {"workload": "config-1 predicate at SF100: l_shipdate < DATE '1994-01-01' -> l_quantity",
                                   "rows_per_gpu": ns, "parallelism": f"row-range shard{world}, no collective"},
                        "roofline": roofline(scan_bytes / ns, ns, float(np.median(scan_steps)),
                                             "filter_mask_tile_kernel<32> + tile_scan + compact_tile_kernel "
                                             "(B200_FILTER_FUSED=1: filter_fused_tile_kernel)", None)}
        # the same predicate with l_shipdate as a DICTIONARY vector (2526 distinct dates + one uint32 index per row, what
        # DuckDB hands over for dictionary-compressed segments): generic expression interpreter (csrc/filter.cu)
        dvals = torch.arange(8036, 8036 + 2526, device=dev, dtype=torch.int32)
        dsel = (shipdate - 8036).to(torch.int32)
        dbatch = ops.Batch.wrap(ctx, [(dvals.data_ptr(), capi.INT32, None, dsel.data_ptr(), 2526),
                                      (quantity.data_ptr(), capi.INT64)], ns, keepalive=[dvals, dsel, quantity])

        def dstep():
            o, cc, _, _ = fp.execute(dbatch)
            dstep.c = cc
            o.free()

        dict_ms = timed_steps(dstep, warmup=2, steps=3)
        assert dstep.c == c, "dictionary-vector scan count mismatch"
        line["scan"]["dictionary_vector"] = {"value": world * ns / (dict_ms / 1e3), "unit": "rows/s", "ms_per_step": dict_ms,
                                             "kernel": "filter_mask_kernel + compact_kernel (generic interpreter: per-row "
                                                       "vector-type dispatch, dictionary gather)",
                                             "achieved_gbs": (ns * 12 + c * 8) / (dict_ms / 1e3) / 1e9}
        del dbatch, dsel
        tm, tc_ = traffic.get("filter_mask"), traffic.get("filter_compact")
        if tm and tc_:
            line["scan"]["roofline"]["traffic"] = int(round((tm["dram_bytes_per_row"] + tc_["dram_bytes_per_row"]) * ns))
            line["scan"]["roofline"]["traffic_source"] = "profiles/r2_filter_mask_ncu.txt + profiles/r2_filter_compact_ncu.txt"

        def check(m, ref_rows):
            o, cc, _, _ = fp.execute(wrap([shipdate, quantity], [capi.INT32, capi.INT64], m))
            from duckdb_b200.distributed import _DevArray
            inf = o.column_info(0)
            got = (int(torch.as_tensor(_DevArray(inf.data, cc, "<i8"), device=dev).sum().item()) if cc else 0, cc)
            o.free()
            want = (int(ref_rows[0][0]), int(ref_rows[0][1]))
            return f"bit-exact on {m} rows (survivor count and sum(l_quantity))" if got == want else f"MISMATCH {got} vs {want}"

        checks["scan"] = check
        checks["_keep_scan"] = (d, sb)

    if "scan" not in skip:
        guarded("scan", leg_scan)

    # ----------------------------------------------------------------- the operators INSIDE DuckDB (libb200_duckdb.so)
    def leg_duckdb():
        """TPC-H Q1 / Q14 shapes through the reference-side binding: the unmodified reference plans the query, the
        optimizer extension swaps in B200HashAggregate / B200HashJoin, DataChunks are staged through pinned morsels.
        Timed next to the stock operators in the SAME connection (B200_DISABLE toggles the optimizer hook)."""
        import ctypes as C

        from oracle import duckdb_ref as R

        ext_path = os.path.join(ROOT, "integration", "_build", "libb200_duckdb.so")
        if not R.available() or not os.path.exists(ext_path):
            line["e2e_duckdb"] = {"unavailable": "needs oracle/_ref/libduckdb_ref.so and integration/_build/libb200_duckdb.so"}
            return
        R.lib()
        ext = C.CDLL(ext_path, mode=C.RTLD_GLOBAL)
        ext.b200_duckdb_register.argtypes = [C.c_void_p]
        cores, _ = BD.effective_cores()
        con = R.Connection(threads=cores)
        assert ext.b200_duckdb_register(con.db) == 0
        sf = args.duckdb_sf
        con.execute(f"CALL dbgen(sf={sf})")
        nli = int(con.fetchall("SELECT count(*) FROM lineitem")[0][0])
        q1 = ("SELECT rf, ls, sum(l_quantity), sum(l_extendedprice), sum(l_extendedprice * (1 - l_discount)), "
              "sum(l_extendedprice * (1 - l_discount) * (1 + l_tax)), avg(l_quantity), avg(l_extendedprice), avg(l_discount), "
              "count(*) FROM (SELECT ascii(l_returnflag)::UTINYINT AS rf, ascii(l_linestatus)::UTINYINT AS ls, * FROM lineitem "
              "WHERE l_shipdate <= DATE '1998-09-02') GROUP BY rf, ls ORDER BY rf, ls")
        # Q14's build side with the PROMO flag materialised (the stock optimizer otherwise pulls the LIKE above the join
        # and the VARCHAR payload keeps the join on the host operator)
        con.execute("CREATE TABLE part_promo AS SELECT p_partkey, (p_type LIKE 'PROMO%')::UTINYINT AS promo FROM part")
        q14 = ("SELECT count(*), sum(l_extendedprice), sum(promo) FROM lineitem JOIN part_promo ON l_partkey = p_partkey")
        cfg1 = "SELECT count(*), sum(l_quantity) FROM lineitem WHERE l_shipdate < DATE '1994-01-01'"

        def run(sql, disable, settings=()):
            if disable:
                os.environ["B200_DISABLE"] = "1"
            else:
                os.environ.pop("B200_DISABLE", None)
            for s_ in settings:
                con.execute(s_)
            plan = "\n".join(str(r[-1]) for r in con.fetchall("EXPLAIN " + sql))
            rows = con.fetchall(sql)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                con.fetchall(sql)
                ts.append(time.perf_counter() - t0)
            os.environ.pop("B200_DISABLE", None)
            return rows, float(np.mean(ts)), plan

        out = {"sf": sf, "lineitem_rows": nli, "threads": cores, "unit": "rows/s"}
        r_gpu, t_gpu, plan = run(q1, False, ["SET perfect_ht_threshold=0"])
        r_hash, t_hash, _ = run(q1, True, ["SET perfect_ht_threshold=0"])
        r_stock, t_stock, _ = run(q1, True, ["RESET perfect_ht_threshold"])
        out["q1"] = {"b200_rows_per_s": nli / t_gpu, "stock_hash_group_by_rows_per_s": nli / t_hash,
                     "stock_plan_rows_per_s": nli / t_stock, "operator_in_plan": "B200_HASH_GROUP_BY" in plan,
                     "same_result": r_gpu == r_hash == r_stock}
        con.execute("SET disabled_optimizers='join_filter_pushdown'")
        j_gpu, tj_gpu, jplan = run(q14, False)
        j_cpu, tj_cpu, _ = run(q14, True)
        out["q14"] = {"b200_rows_per_s": nli / tj_gpu, "stock_rows_per_s": nli / tj_cpu,
                      "operator_in_plan": "B200_HASH_JOIN" in jplan, "same_result": j_gpu == j_cpu}
        # config 1 with STOCK optimizer settings: the predicate is pushed into the scan; B200_SCAN_FILTERS pulls it out
        # into a B200Filter (one H2D + kernel + D2H per 2048-row chunk: PCIe-latency-bound by construction)
        con.execute("SET disabled_optimizers=''")
        os.environ["B200_SCAN_FILTERS"] = "1"
        try:
            f_gpu, tf_gpu, fplan = run(cfg1, False)
        finally:
            os.environ.pop("B200_SCAN_FILTERS", None)
        f_cpu, tf_cpu, _ = run(cfg1, True)
        out["config1_filter"] = {"b200_rows_per_s": nli / tf_gpu, "stock_rows_per_s": nli / tf_cpu,
                                 "operator_in_plan": "B200_FILTER" in fplan and "B200_FILTER(host)" not in fplan,
                                 "same_result": f_gpu == f_cpu,
                                 "note": "B200_SCAN_FILTERS=1: table filters pulled out of the scan into B200Filter"}
        con.close()
        line["e2e_duckdb"] = out

    if "duckdb" not in skip and rank == 0 and world == 1:
        guarded("e2e_duckdb", leg_duckdb)

    # ----------------------------------------------------------------- CPU baseline (reference on host cores)
    if "cpu" not in skip and rank == 0 and world == 1:
        try:
            missing = [k for k in ("q1", "ssb", "q3", "join", "scan") if k not in checks]
            for k in missing:
                checks[k] = (lambda *a, **kw: "leg skipped")
            line["cpu_baseline"] = cpu_baseline_leg(args, checks)
        except Exception as ex:  # the CPU leg must never take the GPU numbers down with it
            import traceback

            traceback.print_exc()
            line["cpu_baseline"] = {"value": None, "unit": "rows/s", "cores": 0, "kind": "reference",
                                    "sample": f"failed: {type(ex).__name__}: {ex}"}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

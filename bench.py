#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its config: rows/sec of join + group-by on the TPC-H Q3 shape at SF100 (config C4).

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One step = the whole operator pipeline of the reference's Q3 physical plan (sqllogictest/test_files/tpch/plans/q3.slt.part:60-76)
    FilterExec(c_mktsegment = BUILDING) -> HashJoinExec RightSemi (c_custkey = o_custkey) over FilterExec(o_orderdate < 1995-03-15)
    -> HashJoinExec Inner (o_orderkey = l_orderkey) over FilterExec(l_shipdate > 1995-03-15)
    -> AggregateExec gby [l_orderkey, o_orderdate, o_shippriority] SUM(l_extendedprice * (100 - l_discount))
over synthetic TPC-H-shaped tables (SF100: customer 15M, orders 150M, lineitem 600M rows; int64 fixed-point money; SURVEY.md §8d C4),
executed as three fused pipelines (dfgpu_pipeline: every table is read once, no intermediate batch touches HBM).
rows/sec = input rows of the three tables / time.

* value    : tables resident in HBM (generated there by the counter-based generators), CUDA events on the launching stream;
             inputs (20.6 GB) exceed L2 (126 MB) so no L2 flush is needed.
* e2e      : the same pipelines through the C ABI with HOST buffers (pinned): H2D of all three tables and D2H of the result rows
             inside the timed region.
* roofline : the dominant kernel (pipe_kernel<aggregate> over lineitem), algorithmic bytes = 28 B per lineitem row (SURVEY.md §8d),
             duration from CUDA events around that kernel; `secondary` carries configs C1 / C2 / C3 with their own fractions.
* cpu_baseline / --impl reference : oracle/ C restatement of the same physical plan (oracle_bench_q3: RepartitionExec(Hash) + partitioned
             JoinHashMap joins + multi-column group table, batch_size 8192), all usable host threads — kind "port": the Rust
             reference cannot be built in this image.
* every timed configuration asserts an order-independent fingerprint of its output at the timed size (a wrong kernel cannot
  produce a number): Q3 vs the CPU arm's fingerprint of the same tables, C2 / C3 vs closed forms over the generators.
* --dump-outputs DIR : the result rows of the last timed step (l_orderkey, o_orderdate, o_shippriority, revenue) as DIR/<column>.npy,
             float64, sorted by the group key; above 64 MB a fixed hash sample of the groups (dump_outputs).  The tables come from
             seeded generators, so two builds run with the same arguments can be compared file for file.
N > 1 (torchrun): weak scaling — every rank owns an SF100 shard of an SF(100 N) database (see q3_multi_gpu below).
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

METRIC = "rows/sec join+groupby (TPC-H Q3 shape: filter x3 -> RightSemi join -> Inner join -> 3-key group-by SUM)"
UNIT = "rows/s"
WORKLOAD = "C4 TPC-H Q3-shaped pipeline, SF{sf:g} per GPU (customer {nc} + orders {no} + lineitem {nl} rows), int64 fixed-point money"
M64 = (1 << 64) - 1
# fingerprint [groups, sum l_orderkey, sum o_orderdate, sum o_shippriority, sum revenue] (mod 2^64) of the SF100 result, seed 1:
# produced independently by oracle_bench_q3 (CPU) and by both GPU paths (fused and operator-by-operator), profiles/README.md r2
Q3_FINGERPRINT_SF100 = [12877494, 3862964181007722, 110988412485, 0, 15758670372586799]


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def usable_threads():
    """threads the CPU arm may really use: the affinity mask, capped by the cgroup CPU quota (a 128-thread barrier loop on an
    8-CPU quota is what made round 1's CPU arm vary 5x between boxes)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def gpu_local_cpus(device):
    """CPUs on the GPU's NUMA node (nvidia-smi topo -m "CPU Affinity" column), or None.  Pinned host buffers are allocated on the node of
    the allocating thread: a staging buffer on the far socket costs PCIe H2D bandwidth."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in out.splitlines():
            parts = line.split()
            if parts and parts[0] == f"GPU{device}":
                for tok in parts[1:]:
                    if tok[0].isdigit() and ("-" in tok or "," in tok) and not tok.startswith("NV"):
                        cpus = set()
                        for rng in tok.split(","):
                            lo, _, hi = rng.partition("-")
                            cpus.update(range(int(lo), int(hi or lo) + 1))
                        return cpus & set(os.sched_getaffinity(0)) or None
    except Exception:
        pass
    return None


def mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 16.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""

    def __init__(self, device=0):
        self.device, self.samples, self.proc = device, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------------------------------
def cpu_q3(sf, threads, runs, warm=1):
    """(per-run seconds list, fingerprint, stage rows) of the CPU restatement on the same generated tables"""
    from oracle import oracle as O
    t = O.q3_generate(sf, seed=1, threads=threads)
    for _ in range(warm):
        O.bench_q3(t, threads)
    secs, fp, st = [], None, None
    for _ in range(runs):
        s, fp, st = O.bench_q3(t, threads)
        secs.append(s)
    rows = len(t["c_custkey"]) + len(t["o_orderkey"]) + len(t["l_orderkey"])
    return secs, fp, st, rows


def cpu_sample_sf(full_sf):
    """largest scale factor the host can hold (inputs 27 B/row + exchange buffers + selection scratch: ~0.5 GB per SF)"""
    avail = mem_available_gb()
    sf = full_sf
    while sf > 1 and sf * 0.55 > avail * 0.6:
        sf /= 2
    return sf


def run_reference(args, rank, world):
    """the reference arm: the CPU restatement of the same physical plan (oracle/, kind "port") on all usable host threads"""
    if rank != 0:
        return
    threads = usable_threads()
    full_sf = float(os.environ.get("DFGPU_Q3_SF", "100"))
    sf = cpu_sample_sf(full_sf)
    secs, fp, st, rows = cpu_q3(sf, threads, max(args.steps, 1), warm=max(1, min(args.warmup, 2)))
    if sf == 100:
        assert fp == Q3_FINGERPRINT_SF100, f"CPU arm fingerprint {fp} != {Q3_FINGERPRINT_SF100}"
    value = rows * len(secs) / sum(secs)
    nc, no, nl = int(150_000 * full_sf), int(1_500_000 * full_sf), int(6_000_000 * full_sf)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(secs), "warmup": args.warmup,
            "ms_per_step": 1000 * sum(secs) / len(secs), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic (counter-based generators, identical tables to the GPU arm)",
            "config": {"workload": WORKLOAD.format(sf=full_sf, nc=nc, no=no, nl=nl), "batch_size": 8192, "partition_mode": "Partitioned",
                       "target_partitions": threads, "sample_scale_factor": sf, "fingerprint": fp, "stages": st},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "median_rows_per_s": rows / float(np.median(secs)), "best_rows_per_s": rows / min(secs), "runs": len(secs),
                             "sample": f"SF{sf:g} ({rows} input rows) per step; oracle/oracle.c oracle_bench_q3: the reference's Q3 physical plan with target_partitions = {threads} "
                                       "(filter + RepartitionExec(Hash) of the three scans, partitioned RightSemi and Inner JoinHashMap joins, 3-column group table), "
                                       "batch_size 8192; tables and exchange buffers resident (pre-faulted) before the clock starts"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# secondary configurations (C2 join, C3 group-by, C1 filter): device resident, each verified at the timed size
# ---------------------------------------------------------------------------------------------------------------------
def splitmix64_np(seed, idx):
    z = (np.uint64(seed) + (idx + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def gen_sum(kind, seed, a, b, n, chunk=1 << 24):
    """wrapping sum of the counter-based generator `kind` over rows [0, n) — closed forms for the secondary fingerprints,
    computed with numpy from the generator DEFINITIONS (include/dfgpu.h dfgpu_gen_kind), independent of any kernel"""
    tot = 0
    with np.errstate(over="ignore"):
        for s in range(0, n, chunk):
            i = np.arange(s, min(n, s + chunk), dtype=np.uint64)
            if kind == "splitmix":
                v = splitmix64_np(seed, i)
            elif kind == "sparse_of":     # splitmix64(seed, splitmix64(a, i) % b)
                v = splitmix64_np(seed, splitmix64_np(a, i) % np.uint64(b))
            else:                          # uniform: a + splitmix64(seed, i) % b
                v = (np.uint64(a & M64) + splitmix64_np(seed, i) % np.uint64(b))
            tot = (tot + int(v.sum(dtype=np.uint64))) & M64
    return tot


def boundary_costs(ctx, D):
    """what the reference-facing boundary costs when the caller does NOT hand over pinned, large batches: FilterExec (x > c, 20 % selected) fed
    (a) one 64M-row batch from pinned / pageable / page-locked-in-place (dfgpu_host_register) host memory, (b) the same rows as 8192-row batches"""
    import ctypes as C
    n = 1 << 26
    nodes = [(D.EXPR_COLUMN, 0, 0, 0, 0, 0.0), (D.EXPR_LITERAL, 0, D.INT64, 0, int((1 << 32) * 0.8), 0.0), (D.EXPR_BINARY, D.OP_GT, 0, 0, 0, 0.0)]
    dx = ctx.generate_i64(D.GEN_UNIFORM, 1, 0, 1 << 32, 0, n)
    pinned = ctx.pinned_empty(n, np.int64)
    ctx.check(ctx.lib.dfgpu_memcpy_d2h(ctx.h, pinned.ctypes.data_as(C.c_void_p), C.c_void_p(dx.ptr), n * 8)); ctx.sync()
    pageable = np.array(pinned, copy=True)
    registered = np.array(pinned, copy=True)
    ctx.check(ctx.lib.dfgpu_host_register(ctx.h, registered.ctypes.data_as(C.c_void_p), registered.nbytes))

    def run(host, batch_rows):
        f = D.FilterHandle(ctx, [D.INT64], nodes, batch_size=8192)
        kept = 0
        for s in range(0, n, batch_rows):
            f.push_host([D.HostColumn(host[s:s + batch_rows])])
            for o in f.drain(host=True):
                kept += o.num_rows; o.release()
        f.finish()
        for o in f.drain(host=True):
            kept += o.num_rows; o.release()
        f.close()
        return kept
    out = {}
    for name, host, br, rows in (("pinned_one_batch", pinned, n, n), ("pageable_one_batch", pageable, n, n), ("registered_in_place_one_batch", registered, n, n),
                                 ("pinned_8192_row_batches", pinned, 8192, 1 << 22)):
        sub = host[:rows]
        run(sub, br)
        t0 = time.perf_counter(); kept = run(sub, br); dt = time.perf_counter() - t0
        out[name] = {"rows_per_s": rows / dt, "h2d_gbs": rows * 8 / dt / 1e9, "rows": rows, "kept": int(kept)}
    ctx.check(ctx.lib.dfgpu_host_unregister(ctx.h, registered.ctypes.data_as(C.c_void_p)))
    dx.free()
    out["note"] = "FilterExec x:int64 > c through dfgpu_filter_push_host + next(host=1), wall clock; 8192-row batches are launch / synchronisation bound (INTEGRATION.md §4: coalesce batches in front of a GPU operator)"
    return out


def q3_decimal_money(ctx, D, Q, cu, orr, li, sf, peak):
    """the headline plan over the reference's real money types (benchmarks/src/tpch/mod.rs:52-122): l_extendedprice, l_discount as
    Decimal128(15,2), sum(l_extendedprice * (1 - l_discount)) as Decimal128(38,4) — 128-bit checked arithmetic per row, two accumulator
    words per group.  The unscaled sums equal the int64 variant's, so the same fingerprint pins it at the timed size."""
    ctx.trim_device_cache()
    dl = Q.decimal_money(ctx, li)
    e0, e1 = ctx.event(), ctx.event()

    def step(keep=False):
        res, st = Q.run_q3_fused(ctx, cu, orr, dl)
        if keep:
            return res, st
        for b in res:
            b.release()
        return None, st
    for _ in range(2):
        step()
    ctx.set_kernel_timing(True); ctx.kernel_time_reset()
    ctx.record(e0)
    for _ in range(5):
        step()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1) / 5
    kms, kn = ctx.kernel_time("pipe:lineitem")
    ctx.set_kernel_timing(False)
    res, st = step(keep=True)
    assert res[0].column(3).type == D.decimal128(38, 4), "SUM over Decimal128(38,4) keeps (38,4)"
    fp = Q.result_fingerprint(ctx, res)
    for b in res:
        b.release()
    if sf == 100:
        assert fp == Q3_FINGERPRINT_SF100, f"Q3 SF100 (Decimal128 money) fingerprint {fp} != {Q3_FINGERPRINT_SF100}"
    nl = dl.rows
    algo = 44.0 * nl                      # lineitem: 8 + 16 + 16 + 4 B per row
    k = kms / max(kn, 1)
    rows = cu.rows + orr.rows + nl
    return {"ms_per_step": ms, "rows_per_s": rows / (ms / 1000.0), "lineitem_kernel_ms": k, "achieved_gbs": algo / (k / 1000.0) / 1e9 if k > 0 else None,
            "frac": algo / (k / 1000.0) / 1e9 / peak if k > 0 else None, "fingerprint": fp, "groups": st["groups"],
            "verified": "group count + wrapping sums of every result column (Decimal128: low word + 3 x high word) == the CPU restatement's fingerprint of the same tables" if sf == 100 else "type check only (fingerprint pinned at SF100)",
            "note": "l_extendedprice, l_discount Decimal128(15,2); sum(l_extendedprice * (Some(1),20,0 - l_discount)) -> Decimal128(38,4): checked i128 arithmetic on the 128-bit interpreter (expr_dec.cuh), i128 add_wrapping as two 64-bit atomics"}


def secondary_configs(ctx, D, peak):
    out = {}
    ctx.trim_device_cache()
    col = lambda buf, n: D.DeviceColumn(ctx, D.INT64, n, buf)
    e0, e1 = ctx.event(), ctx.event()
    # ---- C2: HashJoinExec inner 100M x 10M, sparse unique keys (hashbrown path of the reference), 100 % hit ----
    nb, npr = 10_000_000, 100_000_000
    bk = ctx.generate_i64(D.GEN_SPLITMIX, 42, 0, 0, 0, nb); bp = ctx.generate_i64(D.GEN_SPLITMIX, 7, 0, 0, 0, nb)
    pk = ctx.generate_i64(D.GEN_SPARSE_OF, 42, 43, nb, 0, npr); pp = ctx.generate_i64(D.GEN_SPLITMIX, 8, 0, 0, 0, npr)
    build_cols, probe_cols = [col(bk, nb), col(bp, nb)], [col(pk, npr), col(pp, npr)]

    def join_step(keep=False, ordered=True):
        j = D.HashJoinHandle(ctx, [D.INT64, D.INT64], [D.INT64, D.INT64], [0], [0], [0, 0, 1], [0, 1, 1], ordered_output=ordered)
        j.push_build_device(build_cols); j.finish_build()
        j.push_probe_device(probe_cols); j.finish_probe()
        rows = j.metric("output_rows")
        outs = j.drain(host=False)
        fp = None
        if keep:
            s = [0, 0, 0]
            for b in outs:
                for c in range(3):
                    s[c] = (s[c] + D.column_sum_device(ctx, b.column(c))) & M64
            fp = [rows, (s[0] + 3 * s[1] + 5 * s[2]) & M64]
        for b in outs:
            b.release()
        j.close()
        return rows, fp
    for _ in range(2):
        join_step()
    ctx.set_kernel_timing(True); ctx.kernel_time_reset()
    ctx.record(e0)
    for _ in range(5):
        join_step()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1) / 5
    pms, pn = ctx.kernel_time("join_probe")
    ctx.set_kernel_timing(False)
    rows, fp = join_step(keep=True)
    exp = [npr, (gen_sum("sparse_of", 42, 43, nb, npr) + 3 * gen_sum("sparse_of", 7, 43, nb, npr) + 5 * gen_sum("splitmix", 8, 0, 0, npr)) & M64]
    assert fp == exp, f"C2 join fingerprint {fp} != closed form {exp}"
    algo = 16.0 * nb + 16.0 * npr + 24.0 * npr
    out["C2_join_100Mx10M_sparse_unique"] = {"ms_per_step": ms, "rows_per_s": (nb + npr) / ms * 1e3, "achieved_gbs": algo / ms / 1e6, "frac": algo / ms / 1e6 / peak,
                                             "probe_kernel_ms": pms / max(pn, 1), "probe_kernel_frac": 40.0 * npr / (pms / max(pn, 1)) / 1e6 / peak if pn else None,
                                             "fingerprint": fp, "verified": "rows + sum(k + 3 pb + 5 pp) mod 2^64 == closed form over the generators"}
    # the same join when the consumer ignores row order (ordered_output = 0): radix-partitioned probe, TMA-staged partition pass
    for _ in range(2):
        join_step(ordered=False)
    ctx.set_kernel_timing(True); ctx.kernel_time_reset()
    ctx.record(e0)
    for _ in range(5):
        join_step(ordered=False)
    ctx.record(e1)
    ms_r = ctx.elapsed_ms(e0, e1) / 5
    rp_ms, rp_n = ctx.kernel_time("radix_partition"); pr_ms, pr_n = ctx.kernel_time("join_probe")
    ctx.set_kernel_timing(False)
    rows, fp_r = join_step(keep=True, ordered=False)
    assert fp_r == exp, f"C2 radix join fingerprint {fp_r} != closed form {exp}"
    out["C2_join_100Mx10M_sparse_unique_radix_partitioned"] = {"ms_per_step": ms_r, "rows_per_s": (nb + npr) / ms_r * 1e3, "achieved_gbs": algo / ms_r / 1e6, "frac": algo / ms_r / 1e6 / peak,
                                                               "partition_ms": rp_ms / max(rp_n, 1), "probe_kernel_ms": pr_ms / max(pr_n, 1), "fingerprint": fp_r,
                                                               "note": "ordered_output = 0: probe side radix-partitioned on the top hash bits (TMA bulk loads / stores), per-partition probe with the sub-table L2-resident"}
    ctx.trim_device_cache()   # every block starts from the same allocator state (its warm-up steps refill the cache)
    # ---- C2(ii) with a 10 % hit rate: probe keys drawn from a key set 10x the build side (ordered probe; the misses cost a lookup, no output) ----
    pk10 = ctx.generate_i64(D.GEN_SPARSE_OF, 42, 43, 10 * nb, 0, npr)
    probe10 = [col(pk10, npr), col(pp, npr)]

    def join10(keep=False, mf=False):
        j = D.HashJoinHandle(ctx, [D.INT64, D.INT64], [D.INT64, D.INT64], [0], [0], [0, 0, 1], [0, 1, 1], membership_filter=mf)
        j.push_build_device(build_cols); j.finish_build()
        j.push_probe_device(probe10); j.finish_probe()
        rows = j.metric("output_rows")
        outs = j.drain(host=False)
        fp = None
        if keep:
            s = [0, 0, 0]
            for b in outs:
                for c in range(3):
                    s[c] = (s[c] + D.column_sum_device(ctx, b.column(c))) & M64
            fp = [rows, (s[0] + 3 * s[1] + 5 * s[2]) & M64]
        for b in outs:
            b.release()
        j.close()
        return rows, fp
    for _ in range(2):
        join10()
    ctx.record(e0)
    for _ in range(5):
        join10()
    ctx.record(e1)
    ms10 = ctx.elapsed_ms(e0, e1) / 5
    rows10, fp10 = join10(keep=True)
    with np.errstate(over="ignore"):   # closed form: row i hits iff j_i = splitmix(43, i) % (10 nb) < nb; then k = splitmix(42, j_i), pb = splitmix(7, j_i)
        er, es = 0, 0
        for s0 in range(0, npr, 1 << 24):
            i = np.arange(s0, min(npr, s0 + (1 << 24)), dtype=np.uint64)
            jx = splitmix64_np(43, i) % np.uint64(10 * nb)
            hit = jx < np.uint64(nb)
            er += int(hit.sum())
            es = (es + int(splitmix64_np(42, jx[hit]).sum(dtype=np.uint64)) + 3 * int(splitmix64_np(7, jx[hit]).sum(dtype=np.uint64)) + 5 * int(splitmix64_np(8, i[hit]).sum(dtype=np.uint64))) & M64
    assert fp10 == [er, es], f"C2 10%-hit fingerprint {fp10} != closed form {[er, es]}"
    algo10 = 16.0 * nb + 16.0 * npr + 24.0 * er
    out["C2_join_100Mx10M_sparse_unique_10pct_hit"] = {"ms_per_step": ms10, "rows_per_s": (nb + npr) / ms10 * 1e3, "output_rows": int(rows10), "achieved_gbs": algo10 / ms10 / 1e6,
                                                       "frac": algo10 / ms10 / 1e6 / peak, "fingerprint": fp10, "verified": "rows + checksum == closed form over the generators"}
    # the same with the build keys' membership filter tested before the table (dfgpu_hashjoin_options.membership_filter): 90 % of the probe rows
    # stop at an L2-resident filter word instead of paying a DRAM table access
    for _ in range(2):
        join10(mf=True)
    ctx.record(e0)
    for _ in range(5):
        join10(mf=True)
    ctx.record(e1)
    ms10f = ctx.elapsed_ms(e0, e1) / 5
    rows10f, fp10f = join10(keep=True, mf=True)
    assert fp10f == [er, es], f"C2 10%-hit (membership filter) fingerprint {fp10f} != closed form {[er, es]}"
    out["C2_join_100Mx10M_sparse_unique_10pct_hit_membership_filter"] = {"ms_per_step": ms10f, "rows_per_s": (nb + npr) / ms10f * 1e3, "output_rows": int(rows10f),
                                                                         "achieved_gbs": algo10 / ms10f / 1e6, "frac": algo10 / ms10f / 1e6 / peak, "fingerprint": fp10f,
                                                                         "verified": "rows + checksum == closed form over the generators",
                                                                         "note": "Bloom filter over the build keys (16 bits per key, 20 MB: L2-resident) tested before the 400 MB table — the stand-alone join's dynamic filter pushdown"}
    pk10.free()
    ctx.trim_device_cache()   # every block starts from the same allocator state (its warm-up steps refill the cache)
    # ---- C2(iii): duplicated build keys (the chained table: count -> scan -> emit -> take), ~4 build rows per key, every probe row hits ----
    nk = nb // 4
    bkd = ctx.generate_i64(D.GEN_SPARSE_OF, 42, 99, nk, 0, nb)          # build key of row b = splitmix(42, splitmix(99, b) % nk)
    npd = npr // 4                                                       # 25M probe rows x ~5 matches = ~125M output rows
    pkd = ctx.generate_i64(D.GEN_SPARSE_OF, 42, 43, nk, 0, npd)
    build_d, probe_d = [col(bkd, nb), col(bp, nb)], [col(pkd, npd), col(pp, npd)]

    def joind(keep=False):
        j = D.HashJoinHandle(ctx, [D.INT64, D.INT64], [D.INT64, D.INT64], [0], [0], [0, 0, 1], [0, 1, 1])
        j.push_build_device(build_d); j.finish_build()
        j.push_probe_device(probe_d); j.finish_probe()
        rows = j.metric("output_rows")
        outs = j.drain(host=False)
        fp = None
        if keep:
            s = [0, 0, 0]
            for b in outs:
                for c in range(3):
                    s[c] = (s[c] + D.column_sum_device(ctx, b.column(c))) & M64
            fp = [rows, (s[0] + 3 * s[1] + 5 * s[2]) & M64]
        for b in outs:
            b.release()
        j.close()
        return rows, fp
    for _ in range(2):
        joind()
    ctx.record(e0)
    for _ in range(5):
        joind()
    ctx.record(e1)
    msd = ctx.elapsed_ms(e0, e1) / 5
    rowsd, fpd = joind(keep=True)
    with np.errstate(over="ignore"):   # closed form: multiplicity and payload sum per key slot, then one pass over the probe rows
        ib = np.arange(nb, dtype=np.uint64)
        jb = (splitmix64_np(99, ib) % np.uint64(nk)).astype(np.int64)
        mult = np.bincount(jb, minlength=nk).astype(np.uint64)
        pbv = splitmix64_np(7, ib)
        order = np.argsort(jb, kind="stable"); cs = np.concatenate([[np.uint64(0)], np.cumsum(pbv[order], dtype=np.uint64)])
        starts = np.concatenate([[0], np.cumsum(mult.astype(np.int64))])
        spb = cs[starts[1:]] - cs[starts[:-1]]                           # wrapping sum of pb over the build rows of each key slot
        ip = np.arange(npd, dtype=np.uint64)
        jp = (splitmix64_np(43, ip) % np.uint64(nk)).astype(np.int64)
        m = mult[jp]
        er = int(m.sum())
        es = (int((splitmix64_np(42, jp.astype(np.uint64)) * m).sum(dtype=np.uint64)) + 3 * int(spb[jp].sum(dtype=np.uint64)) + 5 * int((splitmix64_np(8, ip) * m).sum(dtype=np.uint64))) & M64
    assert fpd == [er, es], f"C2 duplicated-build fingerprint {fpd} != closed form {[er, es]}"
    algod = 16.0 * nb + 16.0 * npd + 24.0 * er
    out["C2_join_25Mx10M_duplicated_build_keys_chained"] = {"ms_per_step": msd, "rows_per_s": (nb + npd) / msd * 1e3, "output_rows": int(rowsd), "achieved_gbs": algod / msd / 1e6,
                                                             "frac": algod / msd / 1e6 / peak, "fingerprint": fpd, "verified": "rows + checksum == closed form over the generators",
                                                             "note": "2.5M distinct keys x ~4 build rows each (Poisson), 25M probe rows, every probe row matches its key's whole chain in ascending build row"}
    bkd.free(); pkd.free()
    for b in (bk, bp, pk, pp):
        b.free()
    ctx.trim_device_cache()   # every block starts from the same allocator state (its warm-up steps refill the cache)
    # ---- C3: group-by SUM / COUNT, 1B rows -> 1M groups ----
    ng, gn = 1_000_000, 1_000_000_000
    gk = ctx.generate_i64(D.GEN_UNIFORM, 5, 0, ng, 0, gn); gv = ctx.generate_i64(D.GEN_UNIFORM, 6, -2**31, 2**32, 0, gn)

    def agg_step(keep=False):
        a = D.AggHandle(ctx, [D.INT64, D.INT64], [0], [(D.AGG_SUM, 1, -1), (D.AGG_COUNT, 1, -1)], capacity_hint=ng)
        a.push_device([col(gk, gn), col(gv, gn)]); a.finish()
        g = a.metric("num_groups")
        outs = a.drain(host=False)
        fp = None
        if keep:
            s = [0, 0, 0]
            for b in outs:
                for c in range(3):
                    s[c] = (s[c] + D.column_sum_device(ctx, b.column(c))) & M64
            fp = [g, (3 * s[0] + 5 * s[1] + 7 * s[2]) & M64]
        for b in outs:
            b.release()
        a.close()
        return g, fp
    agg_step()
    ctx.record(e0)
    for _ in range(3):
        agg_step()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1) / 3
    g, fp = agg_step(keep=True)
    # every key 0..ng-1 occurs (1000 rows per group on average), sums and counts are conserved: 3 sum(keys) + 5 sum(v) + 7 n
    exp = [ng, (3 * (ng * (ng - 1) // 2) + 5 * gen_sum("uniform", 6, -2**31, 2**32, gn) + 7 * gn) & M64]
    assert fp == exp, f"C3 group-by fingerprint {fp} != closed form {exp}"
    algo = 16.0 * gn + 24.0 * ng
    out["C3_groupby_sum_count_1B_rows_1M_groups"] = {"ms_per_step": ms, "rows_per_s": gn / ms * 1e3, "groups": int(g), "achieved_gbs": algo / ms / 1e6, "frac": algo / ms / 1e6 / peak,
                                                    "fingerprint": fp, "verified": "groups + (3 sum key + 5 sum sum + 7 sum count) mod 2^64 == closed form over the generators",
                                                    "note": "agg_update_pair_kernel: {sum, count} of a slot share a sector and a lane pair updates them with one RED; the tag bucket is one 256-bit load (DFGPU_AGG_PAIRED=0 for the kernel with one RED per aggregate and row)"}
    gk.free(); gv.free()
    ctx.trim_device_cache()   # every block starts from the same allocator state (its warm-up steps refill the cache)
    # ---- C1 shape: FilterExec x:int64 > c over 100M rows x 2 columns, selectivity 20 % ----
    fn = 100_000_000
    fx = ctx.generate_i64(D.GEN_UNIFORM, 1, 0, 1 << 32, 0, fn); fy = ctx.generate_i64(D.GEN_SPLITMIX, 2, 0, 0, 0, fn)
    lit = int((1 << 32) * 0.8)
    nodes = [(D.EXPR_COLUMN, 0, 0, 0, 0, 0.0), (D.EXPR_LITERAL, 0, D.INT64, 0, lit, 0.0), (D.EXPR_BINARY, D.OP_GT, 0, 0, 0, 0.0)]

    def filter_step(keep=False):
        f = D.FilterHandle(ctx, [D.INT64, D.INT64], nodes, batch_size=0)
        f.push_device([col(fx, fn), col(fy, fn)]); f.finish()
        outs = f.drain(host=False)
        kept = sum(o.num_rows for o in outs)
        fp = [kept, sum(D.column_sum_device(ctx, o.column(0)) for o in outs) & M64] if keep else None
        for o in outs:
            o.release()
        f.close()
        return kept, fp
    filter_step()
    ctx.record(e0)
    for _ in range(3):
        filter_step()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1) / 3
    kept, fp = filter_step(keep=True)
    with np.errstate(over="ignore"):
        ek, es = 0, 0
        for s in range(0, fn, 1 << 24):
            v = splitmix64_np(1, np.arange(s, min(fn, s + (1 << 24)), dtype=np.uint64)) % np.uint64(1 << 32)
            m = v > np.uint64(lit)
            ek += int(m.sum()); es = (es + int(v[m].sum(dtype=np.uint64))) & M64
    assert fp == [ek, es], f"C1 filter fingerprint {fp} != closed form {[ek, es]}"
    fbytes = 16.0 * fn + 16.0 * kept
    out["C1_shape_filter_100M_rows_sel20"] = {"ms_per_step": ms, "rows_per_s": fn / ms * 1e3, "kept": int(kept), "achieved_gbs": fbytes / ms / 1e6, "frac": fbytes / ms / 1e6 / peak,
                                              "fingerprint": fp, "verified": "kept rows + sum(x | x > c) mod 2^64 == numpy over the generator"}
    fx.free(); fy.free()
    return out


RESULT_COLUMNS = ("l_orderkey", "o_orderdate", "o_shippriority", "revenue")
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 0x5EED


def dump_outputs(res, out_dir, max_bytes=DUMP_MAX_BYTES):
    """write the Q3 result rows (the batches a caller of run_q3_fused receives) as out_dir/<column>.npy, float64 (every value here is
    an integer below 2^53, so the conversion is exact; a NULL would be NaN), rows sorted by the group key.  A result larger than max_bytes
    keeps the groups whose splitmix64(DUMP_SEED, l_orderkey) % m == 0 for the smallest m that fits: the same groups whatever order the
    batches came in, so two builds can be compared array for array."""
    cols = [[] for _ in RESULT_COLUMNS]
    for b in res:
        for i, out in enumerate(cols):
            vals, valid = b.column_numpy(i)
            vals = vals.astype(np.float64)
            if valid is not None:
                vals[~valid] = np.nan
            out.append(vals)
    cols = [np.concatenate(c) if c else np.zeros(0, np.float64) for c in cols]
    order = np.lexsort(cols[2::-1])                         # by l_orderkey, then o_orderdate, o_shippriority
    cols = [c[order] for c in cols]
    with np.errstate(over="ignore"):
        h = splitmix64_np(DUMP_SEED, cols[0].astype(np.uint64))
    keep, m = np.ones(len(h), bool), 1
    while keep.sum() * 8 * len(cols) + 128 * len(cols) > max_bytes:       # 128 B: the .npy header of a 1-D array
        m += 1
        keep = h % np.uint64(m) == 0
    os.makedirs(out_dir, exist_ok=True)
    for name, c in zip(RESULT_COLUMNS, cols):
        np.save(os.path.join(out_dir, name + ".npy"), c[keep])
    return int(keep.sum()), m


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result rows of the last timed step as DIR/<column>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the single-GPU result of the CUDA path (--impl ours, one process)")
    if args.impl == "reference":
        return run_reference(args, rank, world)

    from datafusion_b200 import capi as D
    import q3_device_pipeline as Q
    sf = float(os.environ.get("DFGPU_Q3_SF", "100"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        import q3_multi_gpu as QM
        runner = QM.PartitionedQ3(local, dist, sf)
        ctx = runner.ctx
        step = runner.step
        in_rows_rank = runner.input_rows
    else:
        ctx = D.Context(local)
        cu, orr, li = Q.gen_tables(ctx, sf)
        in_rows_rank = cu.rows + orr.rows + li.rows
        last = {}

        def step():
            res, st = Q.run_q3_fused(ctx, cu, orr, li)
            for b in last.get("res", []):
                b.release()
            last["res"], last["st"] = res, st
            return st

    def barrier():
        ctx.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        st = step()
    barrier()
    ctx.set_kernel_timing(True)
    ctx.kernel_time_reset()
    launches0 = ctx.launches + (runner.extra_launches() if world > 1 else 0)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = ctx.event(), ctx.event()
    ctx.record(e0)
    for _ in range(args.steps):
        st = step()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1)
    barrier()
    clk = clocks.stop() if rank == 0 else None
    launches = ctx.launches + (runner.extra_launches() if world > 1 else 0) - launches0
    ktimes = {k: ctx.kernel_time(k) for k in ("pipe:lineitem", "pipe:orders", "pipe:owner_probe_agg", "pipeline_build", "pipeline_output", "lookup_insert", "filter_allreduce",
                                              "partition")}
    ctx.set_kernel_timing(False)
    # ---- the timed output, verified at the timed size ----
    if world > 1:
        import torch
        fp_local = runner.fingerprint()
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        fp_all = runner.all_reduce_fingerprint(fp_local)
        fp = fp_all[:5]
        if rank == 0 and os.environ.get("DFGPU_BENCH_VERIFY", "1") != "0":
            # the timed output at the timed size vs an independent CPU evaluation of the same SF(sf x N) database (streaming regeneration,
            # oracle_q3_stream_fingerprint: no table in memory) — the checker, not the thing measured
            from oracle import oracle as O
            efp, ejoined, equal_orders = O.q3_stream_fingerprint(sf * world, seed=1, threads=usable_threads())
            assert fp == efp and fp_all[5] == ejoined and fp_all[6] == equal_orders, f"multi-GPU Q3 fingerprint {fp_all} != CPU evaluation {efp + [ejoined, equal_orders]}"
    else:
        fp = Q.result_fingerprint(ctx, last["res"])
        if sf == 100:
            assert fp == Q3_FINGERPRINT_SF100, f"Q3 SF100 fingerprint {fp} != {Q3_FINGERPRINT_SF100}"
        if args.dump_outputs:
            dump_outputs(last["res"], args.dump_outputs)
    ms_per_step = ms / args.steps
    in_rows = in_rows_rank * world
    value = in_rows / (ms_per_step / 1000.0)
    nc, no, nl = int(150_000 * sf), int(1_500_000 * sf), int(6_000_000 * sf)

    line = None
    if rank == 0:
        peak, peak_src = peaks()
        a_ms, a_n = ktimes["pipe:lineitem"]      # the lineitem scan: N = 1 filter -> Bloom -> probe -> SUM; N > 1 filter -> membership filter -> output
        k_ms = a_ms / max(a_n, 1)
        algo_bytes = 28.0 * nl                 # lineitem: 8 + 8 + 8 + 4 B per row, every column once (SURVEY.md §8d C4)
        achieved = algo_bytes / (k_ms / 1000.0) / 1e9 if k_ms > 0 else 0.0
        q_bytes = 16.0 * nc + 24.0 * no + 28.0 * nl   # whole pipeline: every input column once (this generator's widths)
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2c_pipeline_traffic.json")))["pipe_kernel_agg_sf100_dram_bytes"]
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": "pipe_kernel<aggregate> (lineitem: filter -> Bloom -> probe -> SUM into the matched record)" if world == 1 else
                    "pipe_kernel<output> (lineitem: filter -> pushed-down membership filter -> survivors to the exchange)", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write at SF100, profiles/r2c_pipeline_traffic.json)",
                    "peak_source": peak_src, "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_per_step, "algorithmic_bytes_per_launch": algo_bytes,
                    "launches_per_step": a_n / args.steps,
                    "whole_pipeline_achieved_gbs": q_bytes / (ms_per_step / 1000.0) / 1e9 if world == 1 else None,
                    "whole_pipeline_frac": q_bytes / (ms_per_step / 1000.0) / 1e9 / peak if world == 1 else None,
                    "other_kernels_ms_per_step": {k: v[0] / args.steps for k, v in ktimes.items() if v[1] and k != "pipe:lineitem"}}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic (generated in HBM, counter-based)",
                "config": {"workload": WORKLOAD.format(sf=sf, nc=nc, no=no, nl=nl), "rows_per_step": in_rows, "stages": st, "fingerprint": fp,
                           "fingerprint_verified": "asserted against the CPU restatement's fingerprint of the same tables" if world == 1 else f"sum over ranks asserted against oracle_q3_stream_fingerprint of the SF{sf * world:g} database",
                           "l2": "inputs (20.6 GB/GPU) exceed L2; no flush",
                           "plan": "3 fused pipelines (dfgpu_pipeline): customer -> key bitmap; orders -> filter + semi probe -> build {o_orderkey -> (o_orderdate, o_shippriority)} + Bloom filter; lineitem -> filter + Bloom + probe + SUM into the matched record" if world == 1 else
                                   "per rank: customer keys all-gathered -> global bitmap; orders -> filter + semi -> membership filter (OR-all-reduced over NVLink) + exchange -> owner builds the join table; lineitem -> filter + membership filter -> exchange -> owner probes + SUMs into the matched record (scripts/q3_multi_gpu.py)",
                           "exchange": "none (single GPU)" if world == 1 else runner.exchange_description()},
                "clocks": clk, "gpu_launches": int(launches), "roofline": roofline}

    # ---- e2e through the C ABI with host (pinned) buffers ----
    if world == 1:
        import ctypes as C
        old_aff = os.sched_getaffinity(0)
        local_cpus = gpu_local_cpus(local)
        if local_cpus:
            os.sched_setaffinity(0, local_cpus)     # allocate (first-touch) the pinned staging buffers on the GPU's NUMA node
        hcols = {}
        for tname, t in (("c", cu), ("o", orr), ("l", li)):
            hs = []
            for c, ty in zip(t.cols, t.types):
                h = ctx.pinned_empty(t.rows, D.NP_OF_TYPE[ty])
                ctx.check(ctx.lib.dfgpu_memcpy_d2h(ctx.h, h.ctypes.data_as(C.c_void_p), C.c_void_p(c.values), t.rows * D.WIDTH[ty]))
                hs.append(h)
            hcols[tname] = hs
        ctx.sync()
        h2d = sum(h.nbytes for hs in hcols.values() for h in hs)

        def e2e_step():
            res, st2, d2h = Q.run_q3_fused_host(ctx, [D.HostColumn(h, None, ty) for h, ty in zip(hcols["c"], cu.types)],
                                                [D.HostColumn(h, None, ty) for h, ty in zip(hcols["o"], orr.types)],
                                                [D.HostColumn(h, None, ty) for h, ty in zip(hcols["l"], li.types)], cu.types, orr.types, li.types)
            return res, st2, d2h
        res, st2, d2h = e2e_step()
        assert st2["groups"] == st["groups"]
        ctx.sync()
        t0 = time.perf_counter()
        for _ in range(max(args.e2e_steps, 1)):
            res, st2, d2h = e2e_step()
        ctx.sync()
        t1 = time.perf_counter()
        args.e2e_steps = max(args.e2e_steps, 1)
        line["e2e"] = {"value": in_rows * args.e2e_steps / (t1 - t0), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps,
                       "ms_per_step": 1000 * (t1 - t0) / args.e2e_steps, "timer": "host wall clock around the C-ABI calls (H2D of the three tables from pinned memory, kernels, D2H of the result rows)",
                       "pcie_gbs": (h2d + d2h) * args.e2e_steps / (t1 - t0) / 1e9, "host_thread_pinned_to_gpu_numa_node": bool(local_cpus)}
        del hcols
        os.sched_setaffinity(0, old_aff)
    elif rank == 0 or world > 1:
        e2e = runner.e2e(args.e2e_steps, barrier)
        if rank == 0:
            line["e2e"] = e2e

    if rank == 0 and world == 1 and not args.no_secondary:
        for b in last.get("res", []):
            b.release()
        last.clear()
        dec_block = None
        try:
            dec_block = q3_decimal_money(ctx, D, Q, cu, orr, li, sf, peak)
        except AssertionError:
            raise
        except Exception as exc:
            dec_block = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        del cu, orr, li          # 20.6 GB of tables: make room for the 16 GB group-by input
        try:
            line["e2e"]["boundary_costs"] = boundary_costs(ctx, D)
        except Exception as exc:
            line["e2e"]["boundary_costs"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            line["roofline"]["secondary"] = secondary_configs(ctx, D, peak)
        except AssertionError:
            raise
        except Exception as exc:
            line["roofline"]["secondary"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        line["roofline"]["secondary"]["C4_q3_decimal128_money"] = dec_block

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            threads = usable_threads()
            csf = cpu_sample_sf(sf)
            secs, cfp, cst, crows = cpu_q3(csf, threads, 3)
            if csf == sf:
                assert cfp == line["config"]["fingerprint"], f"GPU fingerprint {line['config']['fingerprint']} != CPU restatement {cfp}"
            line["cpu_baseline"] = {"value": crows / float(np.median(secs)), "unit": UNIT, "cores": threads, "kind": "port", "best_rows_per_s": crows / min(secs),
                                    "fingerprint": cfp, "same_tables_as_gpu": csf == sf,
                                    "sample": f"SF{csf:g} ({crows} input rows), median of 3 timed runs after one warm-up; oracle_bench_q3 (the reference's Q3 physical plan, target_partitions = {threads}), buffers pre-faulted"}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()

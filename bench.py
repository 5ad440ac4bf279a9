#!/usr/bin/env python
"""bench.py — the hot path on synthetic data, one JSON line (contract: task brief, SURVEY.md §8(d)).

BASELINE.json's metric is "rows/sec hash group_by-agg & join", so the default run measures BOTH halves:
  primary    C2 (configs[1]): hash group_by over 1e8 rows, 1e6 uniform Int64 keys, sum(v_i64)/mean(v_f64)/len
  secondary  C3 (configs[2]): inner hash join 1e8 x 1e7 Int64 — once with dense surrogate keys (the direct-address
             table the library picks for them) and once with SPARSE 64-bit keys, where only the hashed table can serve.
Every workload's result is verified once outside the timed region ("verified" in the line); inputs (>= 0.88 GB) are
larger than L2 (126 MB), so no explicit L2 flush is needed between timed iterations.

  value     rows/s, whole job, inputs resident in HBM when the timed region starts, through the C ABI with BL_DEVICE
            columns (sample + table init + fused build/aggregate + extraction; join: build + probe + emit).
  e2e       the same call with BL_HOST columns in pinned memory: H2D of the inputs and D2H of the result inside the
            timed region.  N > 1: host columns -> device -> the partitioned multi-GPU plan -> host.
  roofline  dominant kernel: algorithmic bytes / its CUDA-event duration on the library stream, against
            MEASURED_PEAKS.json hbm_gbs; kernel_share_of_step for every kernel of the step is in kernels_ms_per_step.
  cpu_baseline  the CPU oracle (C/OpenMP restatement of the reference's partitioned Rayon algorithm, "port") on the
            host cores over a bounded sample, with its 1-thread / 16-thread / all-thread points.

--gpus N (torchrun): weak scaling, every rank owns --rows rows.  group_by: local pre-aggregation, hash partition of the
partial aggregates fused with P2P stores into the owners' windows (counts + flags travel through the windows: no
collective, no host round trip), merge.  join: both relations hash-partitioned (K6) and exchanged with one NCCL
all-to-all-v per relation, local K7/K8, plus the broadcast-build variant.
--impl reference: the oracle on ALL host cores at the full configuration (same rows as the B200 arm).
--dump-outputs DIR: the arrays the last timed step returned, as .npy files named alike in both arms, so that two builds (or the
two arms) can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SPARSE_MULT = np.uint64(0x9E3779B97F4A7C15)      # odd: id -> id * M mod 2^64 is a bijection, so sparse keys stay unique


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "groupby", "join", "q1"])
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--keys", type=int, default=1_000_000)
    ap.add_argument("--build-rows", type=int, default=10_000_000)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=20_000_000, help="rows of the in-line cpu_baseline sample (the --impl reference arm runs the full size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--skew", default="uniform", choices=["uniform", "zipf"], help="group_by key distribution (SURVEY.md 8(d) C2 variants)")
    ap.add_argument("--null-frac", type=float, default=0.0, help="group_by: fraction of null rows in each value column")
    ap.add_argument("--hit-frac", type=float, default=1.0, help="join: fraction of probe rows with a match (C3 variant: 0.5)")
    ap.add_argument("--dup", type=int, default=1, help="join: copies of every build key (C3 variant: 4)")
    ap.add_argument("--join-keys", default="both", choices=["both", "dense", "sparse"], help="join: dense surrogate keys, sparse 64-bit keys, or both")
    ap.add_argument("--acero-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"], help="multi-GPU exchange of the partial aggregates")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed as DIR/<name>.npy "
                    "(float64, nulls as NaN, groups in key order; longer outputs as a fixed, seeded sample of rows, all files together <= 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------- synthetic inputs
def gen_groupby(rows: int, keys: int, seed: int, skew: str = "uniform"):
    """SURVEY.md §8(d) C2: uniform keys (or the Zipf(1.1) variant folded into [0, keys)), v_i64 in
    [-1000,1000), v_f64 = U(0,100).round(6) (h2oai v3)."""
    rng = np.random.default_rng(seed)
    if skew == "zipf":
        key = (rng.zipf(1.1, rows) % keys).astype(np.int64)
    else:
        key = rng.integers(0, keys, rows, dtype=np.int64)
    vi = rng.integers(-1000, 1000, rows, dtype=np.int64)
    vf = rng.uniform(0, 100, rows).round(6)
    return key, vi, vf


def sparsify(ids: np.ndarray) -> np.ndarray:
    """dense ids -> unique sparse 64-bit keys (value range ~2^64: the direct-address table cannot be used)."""
    return (ids.astype(np.uint64) * SPARSE_MULT).view(np.int64)


def gen_join(rows: int, build_rows: int, seed: int, hit_frac: float = 1.0, dup: int = 1, sparse: bool = False, id_base: int = 0, id_space: int | None = None):
    """C3: build = a permutation of [id_base, id_base + build_rows) (unique keys, or `dup` copies of each); probe ids uniform
    over [0, id_space / hit_frac) (id_space = all ranks' build ids under torchrun): 100 % hit by default; variants 50 % hit
    and 4 duplicates per key.  sparse: ids are mapped to unique 64-bit keys by an odd multiplier."""
    rng = np.random.default_rng(seed)
    distinct = max(1, build_rows // dup)
    build = (rng.permutation(distinct * dup).astype(np.int64) % distinct if dup > 1 else rng.permutation(build_rows).astype(np.int64)) + id_base
    space = distinct if id_space is None else id_space
    probe = rng.integers(0, max(1, int(space / hit_frac)), rows, dtype=np.int64)
    if sparse:
        probe, build = sparsify(probe), sparsify(build)
    return probe, build


def gen_lineitem(rows: int, seed: int):
    """BASELINE.json configs[3] (C4): PDS-H / TPC-H lineitem columns used by Q1, synthetic with dbgen-like
    marginals (no dbgen binary here): quantity 1..50, extendedprice = quantity * U(900, 2100), discount
    0..0.10, tax 0..0.08 (2 decimals), returnflag in {A,N,R} / linestatus in {O,F} as dictionary codes,
    shipdate uniform over 1992-01-02 .. 1998-12-01 in days since epoch."""
    rng = np.random.default_rng(seed)
    qty = rng.integers(1, 51, rows).astype(np.float64)
    price = (qty * rng.uniform(900.0, 2100.0, rows)).round(2)
    disc = (rng.integers(0, 11, rows) / 100.0)
    tax = (rng.integers(0, 9, rows) / 100.0)
    ship = rng.integers(8036, 10561, rows).astype(np.int64)            # days: 1992-01-02 .. 1998-12-01
    rf = np.where(ship > 9298, 1, rng.integers(0, 2, rows) * 2).astype(np.int64)   # N after 1995-06-17, else A(0)/R(2)
    ls = (ship > 9298).astype(np.int64)                                  # O(1) / F(0)
    return {"qty": qty, "price": price, "disc": disc, "tax": tax, "ship": ship, "rf": rf, "ls": ls}


Q1_CUTOFF = 10471   # 1998-09-02


def q1_device(plb, d):
    """PDS-H Q1 through the C ABI on device columns: filter (K2+K3) -> expressions (K1) -> group_by/agg (K5)."""
    cols = [d["ship"].view(), d["qty"].view(), d["price"].view(), d["disc"].view(), d["tax"].view(), d["rf"].view(), d["ls"].view()]
    f = plb.filter_cmp(cols, 0, "le", Q1_CUTOFF, location=plb.DEVICE)
    _, qty, price, disc, tax, rf, ls = f
    one_minus = plb.elementwise("sub", np.array([1.0]), disc.view(), location=plb.DEVICE)
    disc_price = plb.elementwise("mul", price.view(), one_minus.view(), location=plb.DEVICE)
    one_plus = plb.elementwise("add", tax.view(), np.array([1.0]), location=plb.DEVICE)
    charge = plb.elementwise("mul", disc_price.view(), one_plus.view(), location=plb.DEVICE)
    key = plb.elementwise("add", plb.elementwise("mul", rf.view(), np.array([256], np.int64), location=plb.DEVICE).view(), ls.view(), location=plb.DEVICE)
    q, p_, dp, ch, di = qty.view(), price.view(), disc_price.view(), charge.view(), disc.view()
    return plb.group_by_agg(key.view(), [("sum", q), ("sum", p_), ("sum", dp), ("sum", ch), ("mean", q), ("mean", p_), ("mean", di), ("len", None)], False, location=plb.DEVICE)


def q1_numpy(h):
    m = h["ship"] <= Q1_CUTOFF
    key = h["rf"][m] * 256 + h["ls"][m]
    dp = h["price"][m] * (1.0 - h["disc"][m])
    ch = dp * (h["tax"][m] + 1.0)
    uk, inv = np.unique(key, return_inverse=True)
    out = {"key": uk, "len": np.bincount(inv)}
    for name, v in (("qty", h["qty"][m]), ("price", h["price"][m]), ("dp", dp), ("ch", ch), ("disc", h["disc"][m])):
        out[name] = np.bincount(inv, weights=v)
    return out


# ------------------------------------------------------------------------------------- verification (outside the timed region)
def verify_groupby(key, vi, vf, val_i, val_f, keys, k, outs) -> str:
    """numpy restatement: bincount over the key ids (sums of +-1000 integers are exact in f64 below 2^53)."""
    if val_i is not None or val_f is not None:
        return "skipped (null variant)"
    o = np.argsort(k, kind="stable")
    uk = np.flatnonzero(np.bincount(key, minlength=keys))
    assert np.array_equal(k[o], uk), "group keys differ from numpy"
    cnt = np.bincount(key, minlength=keys)[uk]
    assert np.array_equal(outs[2][o].astype(np.int64), cnt), "group lengths differ from numpy"
    si = np.bincount(key, weights=vi, minlength=keys)[uk]
    assert np.array_equal(outs[0][o].astype(np.float64), si), "integer sums differ from numpy"
    mf = np.bincount(key, weights=vf, minlength=keys)[uk] / cnt
    assert np.allclose(outs[1][o], mf, rtol=1e-6, atol=0), "means differ from numpy beyond 1e-6 relative"
    return "numpy bincount: keys, len, sum(i64) exact; mean(f64) rtol 1e-6"


def verify_join(probe, build, li, ri, dup) -> str:
    """Exact tuple sequence: every probe row in order, its matches ascending by build row (hash_join/mod.rs:41-50)."""
    order = np.argsort(build, kind="stable")
    sb = build[order]
    lo = np.searchsorted(sb, probe, "left")
    hi = np.searchsorted(sb, probe, "right")
    cnt = hi - lo
    total = int(cnt.sum())
    assert li.size == total and ri.size == total, f"join emitted {li.size} tuples, expected {total}"
    exp_l = np.repeat(np.arange(probe.size, dtype=np.uint32), cnt)
    assert np.array_equal(li, exp_l), "left indices are not the probe rows in order"
    if dup == 1:
        hit = cnt > 0
        assert np.array_equal(ri, order[lo[hit]].astype(np.uint32)), "right indices differ"
    else:
        starts = np.repeat(lo, cnt)
        within = np.arange(total) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        assert np.array_equal(ri, order[starts + within].astype(np.uint32)), "right indices differ (ascending build rows per probe row)"
    return "numpy searchsorted: exact (left_idx, right_idx) sequence"


# ------------------------------------------------------------------------------------- --dump-outputs
DUMP_BYTES = 64_000_000


def by_key(prefix: str, key, cols: dict) -> dict:
    """group_by outputs -> {prefix_key, prefix_<name>: (values, valid)} in ascending key order: the hash group_by returns its groups
    in no fixed order, and sorted they can be compared row for row between runs and builds."""
    o = np.argsort(key[0], kind="stable")
    return {f"{prefix}_{n}": (v[o], None if m is None else np.asarray(m)[o]) for n, (v, m) in {"key": key, **cols}.items()}


def dump_outputs(path: str, outputs: dict, rank: int | None = None):
    """Writes every (values, valid) output as <path>/<name>.npy in float64, NaN where a value is null.  An output longer than its
    share of DUMP_BYTES keeps the rows at positions drawn with a fixed seed, so equal arguments select the same rows every time."""
    os.makedirs(path, exist_ok=True)
    cap = (DUMP_BYTES // len(outputs) - 128) // 8        # 128: the .npy header
    for name, (v, m) in outputs.items():
        if v.size > cap:
            rows = np.sort(np.random.default_rng(0).choice(v.size, cap, replace=False))
            v, m = v[rows], None if m is None else np.asarray(m)[rows]
        out = v.astype(np.float64)
        if m is not None:
            out[~np.asarray(m, bool)] = np.nan
        np.save(os.path.join(path, name + ("" if rank is None else f".rank{rank}") + ".npy"), out)


# ------------------------------------------------------------------------------------- reference arm
def _oracle_threads(oracle):
    hw = oracle.hw_threads()
    oracle.set_threads(hw)          # torchrun exports OMP_NUM_THREADS=1: the port's pool is sized explicitly
    return hw


def _best_threads(oracle, hw: int, run, label: str):
    """The port stands in for a Rayon pool: it is given the thread count it runs FASTEST with on this box (the reference's
    T x N partition scan and a shared, two-socket host make "all hardware threads" the slowest choice here), found on a
    bounded sub-sample before the timed steps."""
    best_t, best_rate, tried = hw, 0.0, []
    for t in sorted({t for t in (8, 16, 32, 64, hw) if t <= hw}):
        oracle.set_threads(t)
        t0 = time.perf_counter()
        n = run(t)
        rate = n / (time.perf_counter() - t0)
        tried.append({"cores": t, "value": rate, "unit": "rows/s"})
        if rate > best_rate:
            best_t, best_rate = t, rate
    oracle.set_threads(best_t)
    return best_t, tried


def run_reference(a):
    import oracle
    oracle.build()
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    hw = _oracle_threads(oracle)
    results = {}
    sub = min(a.rows, 10_000_000)
    if a.workload in ("all", "groupby"):
        key, vi, vf = gen_groupby(a.rows, a.keys, 1, a.skew)
        aggs = [("sum", vi, None), ("mean", vf, None), ("len", None, None)]
        ws = {}

        def gb_probe(t):
            oracle.group_by_agg(key[:sub], None, [(k, None if v is None else v[:sub], m) for k, v, m in aggs], t, False)
            return sub
        tg, tried_g = _best_threads(oracle, hw, gb_probe, "group_by")
        results["groupby"] = ("group_by_agg_rows_per_sec", lambda: oracle.group_by_agg(key, None, aggs, tg, False, workspace=ws), a.rows,
                              f"C2 hash group_by {a.rows} rows, {a.keys} Int64 keys, sum(i64)/mean(f64)/len", tg, tried_g)
    if a.workload in ("all", "join"):
        probe, build = gen_join(a.rows, a.build_rows, 2, a.hit_frac, a.dup, sparse=a.join_keys == "sparse")

        def j_probe(t):
            oracle.hash_join(probe[:sub], build, None, None, "inner", False, "none", t)
            return sub
        tj, tried_j = _best_threads(oracle, hw, j_probe, "join")
        results["join"] = ("hash_join_probe_rows_per_sec", lambda: oracle.hash_join(probe, build, None, None, "inner", False, "none", tj), a.rows,
                           f"C3 inner hash join {a.rows} x {a.build_rows} Int64", tj, tried_j)
    lines, outputs = {}, {}
    for name, (metric, fn, unit_rows, wl, t_used, tried) in results.items():
        oracle.set_threads(t_used)
        for _ in range(min(a.warmup, 1)):
            fn()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            res = fn()
        dt = (time.perf_counter() - t0) / a.steps
        lines[name] = {"metric": metric, "value": unit_rows / dt, "ms_per_step": dt * 1e3, "workload": wl, "cores": t_used, "thread_probe": tried}
        if a.dump_outputs and name == "groupby":
            kout, kv, outs, _ = res
            outputs.update(by_key("groupby", (kout, kv), dict(zip(("sum", "mean", "len"), outs))))
        elif a.dump_outputs:
            tag = "join_sparse" if a.join_keys == "sparse" else "join_dense"
            outputs.update({f"{tag}_left_idx": (res[0], None), f"{tag}_right_idx": (res[1], None)})
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, outputs)
    first = "groupby" if "groupby" in lines else next(iter(lines))
    p = lines[first]
    cores = p["cores"]
    sample = (f"{a.rows} rows/step = the full configuration, on the {cores} of {hw} hardware threads the port runs fastest with (probe on {sub} rows: thread_probe); "
              "oracle = C/OpenMP restatement of the reference's partitioned Rayon algorithm (not Polars itself: no Rust toolchain / wheel)")
    line = {"impl": "reference", "metric": p["metric"], "value": p["value"], "unit": "rows/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": min(a.warmup, 1),
            "ms_per_step": p["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/float64", "data": "synthetic",
            "config": {"workload": p["workload"], "rows_per_step": a.rows, "same_config": True},
            "cpu_baseline": {"value": p["value"], "unit": "rows/s", "cores": cores, "cores_available": hw, "kind": "port", "sample": sample, "thread_probe": p["thread_probe"]},
            "e2e": {"value": p["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if len(lines) > 1:
        line["secondary"] = [{"metric": v["metric"], "value": v["value"], "unit": "rows/s", "ms_per_step": v["ms_per_step"], "cores": v["cores"], "thread_probe": v["thread_probe"],
                              "config": {"workload": v["workload"]}} for k, v in lines.items() if k != first]
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------- B200 arm
class Harness:
    """Timing, clocks, max-over-ranks, profiling around one workload's step functions."""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        import polars_b200 as plb
        self.a, self.torch, self.dist, self.plb = a, torch, dist, plb
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        plb.init(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.ext = torch.cuda.ExternalStream(plb.stream(), device=torch.device("cuda", self.local))
        self.peak_gbs, self.peak_src = peaks()
        self.total_launches = 0
        self.clock_rows = []

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()
        self.plb.sync()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: int) -> int:
        if self.world == 1:
            return int(x)
        t = self.torch.tensor([int(x)], dtype=self.torch.int64, device="cuda")
        self.dist.all_reduce(t)
        return int(t.item())

    def measure(self, step_device, step_e2e, unit_rows, alg_bytes_per_row, dominant_pick, traffic_key):
        """-> dict(value, ms_per_step, roofline, kernels_ms_per_step, e2e, clocks, n_out)."""
        a, plb, torch = self.a, self.plb, self.torch
        for _ in range(max(a.warmup, 3)):
            n_out = step_device()
        self.barrier()
        plb.profile_reset()
        plb.profile_enable(True)
        sampler = ClockSampler(self.local)
        if self.rank == 0:
            sampler.start()
        with torch.cuda.stream(self.ext):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                n_out = step_device()
            e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        prof = plb.profile()
        self.total_launches += plb.launch_count()
        plb.profile_enable(False)
        ms_per_step = self.max_over_ranks(ms) / a.steps
        value = unit_rows * self.world / (ms_per_step / 1e3)
        # ---- end to end with pinned host buffers (H2D + compute + D2H per step)
        e2e_vals, d2h = [], 0
        for i in range(a.e2e_steps + 1 if (a.e2e_steps > 0 and step_e2e is not None) else 0):
            self.barrier()
            t0 = time.perf_counter()
            _, d2h = step_e2e()
            dt = time.perf_counter() - t0
            if i > 0:
                e2e_vals.append(dt)
        e2e_s = self.max_over_ranks(float(np.mean(e2e_vals)) if e2e_vals else 0.0)
        clocks = sampler.stop() if self.rank == 0 else None      # sampled over the timed region and the e2e steps that follow it
        dominant = dominant_pick(prof)
        traffic = None      # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of this workload
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get(traffic_key, {}).get(dominant)
        except Exception:
            pass
        dom = prof.get(dominant, {"launches": 0, "ms": 0.0})
        dom_ms = dom["ms"] / max(dom["launches"], 1)
        achieved = (alg_bytes_per_row * unit_rows / 1e9) / (dom_ms / 1e3) if dom_ms > 0 else 0.0
        total_kernel_ms = sum(v["ms"] for v in prof.values()) / a.steps
        per_step = {k: v["ms"] / a.steps for k, v in prof.items()}
        return {"value": value, "ms_per_step": ms_per_step, "n_out": int(n_out),
                "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": self.peak_gbs, "unit": "GB/s", "frac": achieved / self.peak_gbs if self.peak_gbs else None,
                             "traffic": traffic, "peak_source": self.peak_src, "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": alg_bytes_per_row * unit_rows,
                             "kernel_share_of_step": (dom_ms * dom["launches"] / a.steps / total_kernel_ms) if total_kernel_ms else None,
                             "kernel_shares": {k: v / total_kernel_ms for k, v in per_step.items()} if total_kernel_ms else None},
                "kernels_ms_per_step": per_step,
                "e2e": {"value": unit_rows * self.world / e2e_s if e2e_s else None, "unit": "rows/s", "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3},
                "clocks": clocks}


def bench_groupby(H: Harness):
    a, plb, world, rank = H.a, H.plb, H.world, H.rank
    key, vi, vf = gen_groupby(a.rows, a.keys, 1 + rank, a.skew)
    hkey, hvi, hvf = (plb.to_pinned(key), plb.to_pinned(vi), plb.to_pinned(vf)) if a.e2e_steps > 0 else (None, None, None)
    val_i = val_f = None
    if a.null_frac > 0:      # the "+5 % nulls" variant: independent validity bitmaps on both value columns
        nrng = np.random.default_rng(100 + rank)
        val_i, val_f = (plb.pack_bits(nrng.random(a.rows) >= a.null_frac) for _ in range(2))      # Arrow LSB bitmaps
    dkey, dvi, dvf = plb.to_device(key), plb.to_device(vi, val_i), plb.to_device(vf, val_f)
    spec = [("sum", np.int64), ("mean", np.float64), ("len", None)]
    nullable = [val_i is not None, val_f is not None, False]
    peer_ex = None
    pdist = None
    if world > 1:
        from polars_b200 import dist as pdist
        torch, dist = H.torch, H.dist
        if a.exchange == "p2p":      # window region per source rank: every group of a rank could go to one peer
            try:
                peer_ex = pdist.PeerExchange(plb, rows_per_src=min(a.keys, a.rows) + 1024, row_words=2 + 3 + sum(nullable[:2]))
                ok_all = torch.tensor([1], device="cuda")
            except Exception as e:      # CUDA IPC unavailable (container policy): use the NCCL all-to-all instead
                print(f"[bench] peer windows unavailable ({e}); falling back to --exchange nccl", file=sys.stderr)
                ok_all = torch.tensor([0], device="cuda")
            dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
            if int(ok_all.item()) == 0:
                a.exchange, peer_ex = "nccl", None

    def plan(kc, ic, fc, location):
        """One step of the multi-GPU plan on device columns -> (key, [sum, mean, len]) at `location`."""
        vals = [ic, fc, None]
        if a.exchange == "p2p":
            return pdist.partitioned_group_by_p2p(plb, peer_ex, kc, vals, spec, nullable=nullable, location=location)
        return pdist.partitioned_group_by(plb, kc, vals, spec, nullable=nullable, location=location)

    last = {}

    def step_device():
        if world == 1:
            ok, outs = plb.group_by_agg(dkey.view(), [("sum", dvi.view()), ("mean", dvf.view()), ("len", None)], False, location=plb.DEVICE)
        else:
            ok, outs = plan(dkey.view(), dvi.view(), dvf.view(), plb.DEVICE)
        if a.dump_outputs:
            last["out"] = ok, outs
        return ok.length

    def step_e2e():
        if world == 1:
            (k, _), outs = plb.group_by_agg(plb.Column(hkey), [("sum", plb.Column(hvi, val_i)), ("mean", plb.Column(hvf, val_f)), ("len", None)], False, location=plb.HOST)
            return k.size, k.nbytes + sum(o[0].nbytes for o in outs)
        # host -> device -> partitioned plan (exchange over NVLink) -> host
        ck, ci, cf = plb.to_device(hkey), plb.to_device(hvi, val_i), plb.to_device(hvf, val_f)
        ok, outs = plan(ck.view(), ci.view(), cf.view(), plb.DEVICE)
        res = [ok.to_numpy()[0]] + [o.to_numpy()[0] for o in outs]
        return res[0].size, sum(r.nbytes for r in res)

    verified = None
    if not a.no_verify:
        if world == 1:
            (k, _), outs = plb.group_by_agg(dkey.view(), [("sum", dvi.view()), ("mean", dvf.view()), ("len", None)], False, location=plb.HOST)
            verified = verify_groupby(key, vi, vf, val_i, val_f, a.keys, k, [o[0] for o in outs])
        else:
            ok, outs = plan(dkey.view(), dvi.view(), dvf.view(), plb.DEVICE)
            k = ok.to_numpy()[0]; s = outs[0].to_numpy()[0]; ln = outs[2].to_numpy()[0]
            # conservation across ranks + ownership: every group exactly once, on the rank its key hashes to
            h = (k.view(np.uint64) * np.uint64(0x55fbfd6bfc5458e9))
            # hash_to_partition = (h * P) >> 64, exactly, from 32-bit halves: (hi * P + ((lo * P) >> 32)) >> 32
            hi, lo = h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)
            part = ((hi * np.uint64(world) + ((lo * np.uint64(world)) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)
            assert (part == rank).all(), "a group sits on the wrong rank"
            assert H.sum_over_ranks(int(ln.astype(np.int64).sum())) == a.rows * world, "rows lost or duplicated across ranks"
            assert H.sum_over_ranks(int(s.sum())) == H.sum_over_ranks(int(vi.sum())), "integer sums not conserved across ranks"
            groups = H.sum_over_ranks(k.size)
            if a.skew == "uniform" and a.rows * world >= 20 * a.keys:
                assert groups == a.keys, f"{groups} groups over all ranks, expected {a.keys}"
            verified = "conservation over all ranks: rows, sum(i64), group count; ownership by hash_to_partition"
    del key, vi, vf

    def pick(prof):
        return max((k for k in prof if k.startswith("k5_groupby_agg")), key=lambda k: prof[k]["ms"], default="k5_groupby_agg")

    r = H.measure(step_device, step_e2e if a.e2e_steps > 0 else None, a.rows, 24.0, pick, f"groupby:{a.rows}:{a.keys}")
    r["e2e"]["h2d_bytes_per_step"] = int(a.rows * 24)
    r["e2e"]["path"] = ("bl_groupby_agg with BL_HOST columns in pinned memory -> BL_HOST outputs" if world == 1 else
                        "pinned host columns -> bl_column_to(device) -> partitioned plan (local K5, fused partition + P2P exchange, merge) -> host outputs")
    r["metric"] = "group_by_agg_rows_per_sec"
    r["verified"] = verified
    if a.dump_outputs:
        ok, outs = last["out"]
        r["outputs"] = by_key("groupby", ok.to_numpy(), {n: o.to_numpy() for n, o in zip(("sum", "mean", "len"), outs)})
    r["workload"] = (f"C2 hash group_by {a.rows} rows/GPU, {a.keys} {'Zipf(1.1)-skewed' if a.skew == 'zipf' else 'uniform'} Int64 keys, sum(v_i64)/mean(v_f64)/len"
                     + (f", {a.null_frac:.0%} nulls per value column" if a.null_frac > 0 else "") + "; inputs 2.4 GB > L2 (no flush needed)")
    r["parallelism"] = ("single GPU" if world == 1 else
                        (f"hash-partitioned x{world}: local pre-agg + fused partition/P2P-store exchange over NVLink (counts + flags in the peer windows, no host round trip) + merge"
                         if a.exchange == "p2p" else f"hash-partitioned x{world}: local pre-agg + one NCCL all-to-all of partial aggregates + merge"))
    if peer_ex is not None:
        peer_ex.close()
    return r


def bench_join(H: Harness, sparse: bool):
    a, plb, world, rank = H.a, H.plb, H.world, H.rank
    probe, build = gen_join(a.rows, a.build_rows, 2 + rank, a.hit_frac, a.dup, sparse=sparse, id_base=rank * a.build_rows, id_space=None if world == 1 else a.build_rows * world)
    hp, hb = (plb.to_pinned(probe), plb.to_pinned(build)) if a.e2e_steps > 0 else (None, None)
    dp, db = plb.to_device(probe), plb.to_device(build)
    pdist = None
    if world > 1:
        from polars_b200 import dist as pdist

    plan = "single GPU" if world == 1 else pdist.choose_join_plan(a.rows, a.build_rows, world)

    def run_plan(which, pc, bc):
        """One step of a multi-GPU join plan on device key columns -> (left, right) global row-id columns."""
        if which == "broadcast":
            return pdist.broadcast_hash_join(plb, pc, bc, rank * a.rows)
        return pdist.partitioned_hash_join(plb, pc, bc, rank * a.rows, rank * a.build_rows)

    last = {}

    def step_device():
        if world == 1:
            li, ri = plb.hash_join(dp.view(), db.view(), "inner", False, "none", location=plb.DEVICE)
        else:
            li, ri = run_plan(plan, dp.view(), db.view())
        if a.dump_outputs:
            last["out"] = li, ri
        return li.length

    def step_e2e():
        if world == 1:
            (li, _), (ri, _) = plb.hash_join(plb.Column(hp), plb.Column(hb), "inner", False, "none", location=plb.HOST)
            return li.size, li.nbytes + ri.nbytes
        cp, cb = plb.to_device(hp), plb.to_device(hb)
        gl, gr = run_plan(plan, cp.view(), cb.view())
        l, r_ = gl.to_numpy()[0], gr.to_numpy()[0]
        return l.size, l.nbytes + r_.nbytes

    verified = None
    if not a.no_verify:
        if world == 1:
            (li, _), (ri, _) = plb.hash_join(dp.view(), db.view(), "inner", False, "none", location=plb.HOST)
            verified = verify_join(probe, build, li, ri, a.dup)
        else:
            gl, gr = run_plan(plan, dp.view(), db.view())
            n_pairs = H.sum_over_ranks(gl.length)
            exp = a.rows * world * a.dup if a.hit_frac >= 1.0 else None
            assert exp is None or n_pairs == exp, f"{n_pairs} join tuples over all ranks, expected {exp}"
            # global ids -> every emitted left id is a distinct probe row (unique build keys): checked through the id sum
            l = gl.to_numpy()[0].astype(np.int64)
            if a.dup == 1 and a.hit_frac >= 1.0:
                tot = H.sum_over_ranks(int(l.sum()))
                nn = a.rows * world
                assert tot == nn * (nn - 1) // 2, "the emitted probe rows are not each probe row exactly once"
            verified = "conservation over all ranks: tuple count, every probe row exactly once (id sum)"
    del probe, build

    def pick(prof):
        return max((k for k in prof if k.startswith("k8_") and "probe" in k), key=lambda k: prof[k]["ms"], default="k8_join_probe_emit")

    alg = 8.0 + 8.0 * a.hit_frac * a.dup      # probe key + (left_idx, right_idx) u32 per match
    r = H.measure(step_device, step_e2e if a.e2e_steps > 0 else None, a.rows, alg, pick, f"join:{'sparse' if sparse else 'dense'}:{a.rows}:{a.build_rows}")
    r["e2e"]["h2d_bytes_per_step"] = int((a.rows + a.build_rows) * 8)
    r["e2e"]["path"] = ("bl_hash_join with BL_HOST columns in pinned memory -> BL_HOST index columns" if world == 1 else
                        f"pinned host key columns -> device -> {plan} join plan -> global (left, right) row ids on the host")
    r["metric"] = "hash_join_probe_rows_per_sec"
    r["verified"] = verified
    if a.dump_outputs:
        tag = "join_sparse" if sparse else "join_dense"
        r["outputs"] = {f"{tag}_left_idx": last["out"][0].to_numpy(), f"{tag}_right_idx": last["out"][1].to_numpy()}
    r["workload"] = (f"C3 inner hash join: probe {a.rows} x build {a.build_rows} Int64 keys per GPU ({'unique' if a.dup == 1 else str(a.dup) + ' copies of each'}; "
                     f"{'sparse 64-bit values -> hashed table' if sparse else 'dense surrogate ids -> direct-address table'}), {a.hit_frac:.0%} hit; outputs (left_idx,right_idx) u32")
    names = {"partitioned": f"radix hash-partitioned x{world}: K6 on both relations + one NCCL all-to-all-v per relation + local build/probe + K4 to global ids",
             "broadcast": f"broadcast build side x{world}: all-gather of the {a.build_rows * world} build keys (NCCL), probe rows stay local, local build/probe"}
    r["parallelism"] = "single GPU" if world == 1 else names[plan] + " (chosen by the exchange-volume rule, dist.choose_join_plan)"
    if world > 1:
        # the other plan, measured beside the chosen one (BASELINE configs[2] names the radix-partitioned exchange)
        other = "partitioned" if plan == "broadcast" else "broadcast"

        def step_other():
            gl, gr = run_plan(other, dp.view(), db.view())
            return gl.length
        try:
            rb = H.measure(step_other, None, a.rows, alg, pick, "join:" + other)
            r["alternative_plan"] = {"value": rb["value"], "unit": "rows/s", "ms_per_step": rb["ms_per_step"], "kernels_ms_per_step": rb["kernels_ms_per_step"], "parallelism": names[other]}
        except Exception as e:      # optional evidence: never lose the line
            r["alternative_plan"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    return r


def bench_q1(H: Harness):
    a, plb, rank = H.a, H.plb, H.rank
    rows = a.rows if a.rows != 100_000_000 else 60_000_000      # SF10 lineitem ~ 6e7 rows
    h = gen_lineitem(rows, 4 + rank)
    d = {k: plb.to_device(v) for k, v in h.items()}
    hp = {k: plb.to_pinned(v) for k, v in h.items()}
    exp = q1_numpy(h)
    ok, outs = q1_device(plb, d)
    k, _ = ok.to_numpy(); o = np.argsort(k)
    assert np.array_equal(k[o], exp["key"]) and np.array_equal(outs[7].to_numpy()[0][o], exp["len"]), "Q1 groups differ"
    for i, nm in ((0, "qty"), (1, "price"), (2, "dp"), (3, "ch")):
        assert np.allclose(outs[i].to_numpy()[0][o], exp[nm], rtol=1e-6), "Q1 sums differ: " + nm
    del h
    last = {}

    def step_device():
        ok, outs = q1_device(plb, d)
        if a.dump_outputs:
            last["out"] = ok, outs
        return ok.length

    def step_e2e():
        dd = {k: plb.to_device(v) for k, v in hp.items()}
        ok, outs = q1_device(plb, dd)
        res = [ok.to_numpy()[0]] + [o.to_numpy()[0] for o in outs]
        return res[0].size, sum(r.nbytes for r in res)

    def pick(prof):
        return max((k for k in prof if k.startswith("k5_groupby_agg")), key=lambda k: prof[k]["ms"], default="k5_groupby_agg_smem")

    r = H.measure(step_device, step_e2e if a.e2e_steps > 0 else None, rows, 8.0 * 6, pick, f"q1:{rows}")
    r["e2e"]["h2d_bytes_per_step"] = int(rows * 8 * 7)
    r["e2e"]["path"] = "pinned host lineitem columns -> device -> filter + expressions + group_by -> host"
    r["metric"] = "pdsh_q1_rows_per_sec"
    r["verified"] = "numpy: groups, len exact; sums rtol 1e-6"
    if a.dump_outputs:
        ok, outs = last["out"]
        names = ("sum_qty", "sum_price", "sum_disc_price", "sum_charge", "mean_qty", "mean_price", "mean_disc", "len")
        r["outputs"] = by_key("q1", ok.to_numpy(), {n: o.to_numpy() for n, o in zip(names, outs)})
    r["workload"] = f"C4 PDS-H Q1 shape on {rows} synthetic lineitem rows (SF10-sized): filter + 4 expressions + group_by(returnflag,linestatus) with 8 aggregates"
    r["parallelism"] = "single GPU"
    r["rows"] = rows
    return r


def main():
    a = parse()
    sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark caches nothing beside the sources
    # NCCL prints its version banner to STDOUT for any NCCL_DEBUG level: route it to a file so the JSON line stays alone on stdout.
    # The directory is shared by the ranks of one torchrun (their common parent) and lies outside the tree.
    if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
        log_dir = os.path.join(tempfile.gettempdir(), f"bench_nccl_debug.{os.getppid()}")
        os.makedirs(log_dir, exist_ok=True)
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(log_dir, "nccl_debug.%h.%p.log")
    if a.acero_child:
        acero_child(a)
        return
    if a.impl == "reference":
        run_reference(a)
        return
    H = Harness(a)
    results = []
    if a.workload in ("all", "groupby"):
        results.append(bench_groupby(H))
    if a.workload in ("all", "join"):
        if a.join_keys in ("both", "dense"):
            results.append(bench_join(H, sparse=False))
        if a.join_keys in ("both", "sparse"):
            results.append(bench_join(H, sparse=True))
    if a.workload == "q1":
        results.append(bench_q1(H))
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {n: c for r in results for n, c in r.pop("outputs").items()}, H.rank if H.world > 1 else None)
    if H.rank != 0:
        if H.world > 1:
            H.dist.destroy_process_group()
        return
    p = results[0]

    def cfg(r):
        return {"workload": r["workload"], "rows_per_gpu": r.get("rows", a.rows), "rows_out": r["n_out"], "l2_policy": "inputs larger than L2", "parallelism": r["parallelism"]}

    line = {
        "metric": p["metric"], "value": p["value"], "unit": "rows/s", "n_gpus": H.world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": p["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/float64", "data": "synthetic",
        "config": cfg(p), "verified": p["verified"], "roofline": p["roofline"], "kernels_ms_per_step": p["kernels_ms_per_step"],
        "gpu_launches": int(H.total_launches), "clocks": p["clocks"],
        "knobs": {k: v for k, v in os.environ.items() if k.startswith("BL_")},
        "e2e": p["e2e"],
    }
    if len(results) > 1:
        line["secondary"] = [{"metric": r["metric"], "value": r["value"], "unit": "rows/s", "ms_per_step": r["ms_per_step"], "config": cfg(r), "verified": r["verified"],
                              "roofline": r["roofline"], "kernels_ms_per_step": r["kernels_ms_per_step"], "e2e": r["e2e"], "clocks": r["clocks"],
                              **({"alternative_plan": r["alternative_plan"]} if "alternative_plan" in r else {})} for r in results[1:]]
    if H.world == 1 and not a.no_cpu_baseline and a.workload in ("all", "groupby", "join"):
        line["cpu_baseline"] = cpu_baseline(a)
    print(json.dumps(line), flush=True)
    if H.world > 1:
        H.dist.destroy_process_group()
        nccl_debug_summary()


def nccl_debug_summary():
    """NCCL_DEBUG goes to NCCL_DEBUG_FILE (its banner would otherwise land on stdout beside the JSON line); the lines that
    say how the communicator was built (ranks, NVLS / P2P transport) are repeated on stderr for whoever reads the log."""
    pat = os.environ.get("NCCL_DEBUG_FILE")
    if not pat or not os.environ.get("NCCL_DEBUG"):
        return
    import glob
    seen = 0
    for path in sorted(glob.glob(os.path.join(os.path.dirname(pat), "nccl_debug.*.log"))):
        try:
            with open(path) as f:
                for ln in f:
                    if any(t in ln for t in ("nranks", "NVLS", "via P2P", "Init COMPLETE")) and seen < 40:
                        print("[nccl] " + ln.rstrip(), file=sys.stderr)
                        seen += 1
        except OSError:
            pass


def acero_child(a):
    """Child process of `acero_baseline`: times the query on pyarrow's Acero engine and prints one JSON object."""
    import pyarrow as pa
    if a.workload in ("all", "groupby"):
        key, vi, vf = gen_groupby(a.rows, a.keys, 1, a.skew)
        t = pa.table({"key": key, "vi": vi, "vf": vf})
        t0 = time.perf_counter()
        t.group_by("key", use_threads=True).aggregate([("vi", "sum"), ("vf", "mean"), ([], "count_all")])
        dt = time.perf_counter() - t0
    else:
        probe, build = gen_join(a.rows, a.build_rows, 2, a.hit_frac, a.dup)
        lt, rt = pa.table({"key": probe}), pa.table({"key": build, "r": np.arange(build.size, dtype=np.int64)})
        t0 = time.perf_counter()
        lt.join(rt, keys="key", join_type="inner", use_threads=True)
        dt = time.perf_counter() - t0
    print(json.dumps({"engine": f"pyarrow-acero {pa.__version__}", "value": a.rows / dt, "unit": "rows/s", "threads": pa.cpu_count()}), flush=True)
    os._exit(0)      # Acero's worker threads occasionally abort the interpreter during static destruction


def acero_baseline(a, workload: str, sample: int, build_rows: int):
    """Second, independent CPU reference (SURVEY.md 8(d)): the same query on pyarrow's Acero engine with
    its default thread pool, in a child process.  Reported beside the oracle port; neither is the target."""
    cmd = [sys.executable, os.path.abspath(__file__), "--acero-child", "--workload", workload, "--rows", str(sample), "--keys", str(a.keys),
           "--build-rows", str(build_rows), "--skew", a.skew, "--hit-frac", str(a.hit_frac), "--dup", str(a.dup)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:      # optional evidence, never a reason to lose the bench line
        return {"engine": "pyarrow-acero", "unavailable": f"{type(e).__name__}: {e}"[:160]}


def cpu_baseline(a):
    """The oracle port on the host cores over a bounded sample (about 10-30 s of CPU work in total), with its thread
    scaling points.  The full-size number is the --impl reference arm."""
    import oracle
    oracle.build()
    hw = _oracle_threads(oracle)
    sample = min(a.rows, a.cpu_sample)
    points = sorted({t for t in (1, 8, 16, 32, 64, hw) if t <= hw})
    out = {}
    if a.workload in ("all", "groupby"):
        key, vi, vf = gen_groupby(sample, a.keys, 1, a.skew)
        aggs = [("sum", vi, None), ("mean", vf, None), ("len", None, None)]
        scal = []
        for t in points:
            oracle.set_threads(t)
            n = sample if t > 1 else min(sample, 5_000_000)
            t0 = time.perf_counter()
            oracle.group_by_agg(key[:n], None, [(k, None if v is None else v[:n], m) for k, v, m in aggs], t, False)
            scal.append({"cores": t, "value": n / (time.perf_counter() - t0), "unit": "rows/s", "sample": f"{n} rows"})
        oracle.set_threads(hw)
        best = max(scal, key=lambda s: s["value"])
        out = {"value": best["value"], "unit": "rows/s", "cores": best["cores"], "kind": "port",
               "sample": f"{sample} rows of the C2 workload, one pass per point; oracle = C/OpenMP restatement of the reference's partitioned algorithm (the Rust reference cannot be built here)",
               "thread_scaling": scal, "second_reference": acero_baseline(a, "groupby", sample, a.build_rows)}
    if a.workload in ("all", "join"):
        build_rows = max(1, int(a.build_rows * sample / a.rows))
        probe, build = gen_join(sample, build_rows, 2, a.hit_frac, a.dup)
        scal = []
        for t in points:
            oracle.set_threads(t)
            n = sample if t > 1 else min(sample, 5_000_000)
            t0 = time.perf_counter()
            oracle.hash_join(probe[:n], build, None, None, "inner", False, "none", t)
            scal.append({"cores": t, "value": n / (time.perf_counter() - t0), "unit": "rows/s", "sample": f"{n} probe rows x {build_rows} build rows"})
        oracle.set_threads(hw)
        best = max(scal, key=lambda s: s["value"])
        j = {"metric": "hash_join_probe_rows_per_sec", "value": best["value"], "unit": "rows/s", "cores": best["cores"], "kind": "port", "thread_scaling": scal,
             "second_reference": acero_baseline(a, "join", sample, build_rows)}
        if out:
            out["join"] = j
        else:
            out = {**j, "sample": f"{sample} probe rows of the C3 workload"}
    return out


if __name__ == "__main__":
    main()

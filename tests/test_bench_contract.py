"""bench.py's output: the reference arm runs on the CPU, so its JSON line is checked without a GPU — one line, the
expected keys, the `impl: reference` / `cpu_baseline` / `e2e` shape, and that the C2 / C3 variants flags are accepted.
--dump-outputs is checked on the reference arm and, with a GPU, the B200 arm's dump against the reference arm's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ("--rows", "200000", "--keys", "1000", "--build-rows", "20000")
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
        "cpu_baseline", "e2e"}


def run_bench(*args, impl="reference"):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--steps", "1", "--warmup", "1", *SMALL, *args],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, f"expected ONE JSON line on stdout, got {len(lines)}"
    return json.loads(lines[0])


@pytest.mark.parametrize("args,metric", [((), "group_by_agg_rows_per_sec"), (("--workload", "groupby", "--skew", "zipf"), "group_by_agg_rows_per_sec"),
                                         (("--workload", "join", "--hit-frac", "0.5", "--dup", "4"), "hash_join_probe_rows_per_sec")])
def test_reference_arm_line(args, metric):
    d = run_bench(*args)
    assert KEYS <= set(d), sorted(KEYS - set(d))
    assert d["impl"] == "reference" and d["metric"] == metric and d["unit"] == "rows/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["same_config"] is True and d["config"]["rows_per_step"] == 200000
    if not args:      # the default run covers both halves of BASELINE.json's metric: group_by primary, join secondary
        assert [x["metric"] for x in d["secondary"]] == ["hash_join_probe_rows_per_sec"] and d["secondary"][0]["value"] > 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--rows", "100000", "--keys", "1000", "--build-rows", "10000"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs: equal arguments give equal files, and they hold what the seeded workloads compute (numpy restatement)."""
    dumps = []
    for run in ("a", "b"):
        run_bench("--dump-outputs", str(tmp_path / run))
        dumps.append(_load(tmp_path / run))
    d = dumps[0]
    assert sorted(d) == ["groupby_key", "groupby_len", "groupby_mean", "groupby_sum", "join_dense_left_idx", "join_dense_right_idx"]
    for name, x in d.items():
        assert x.dtype == np.float64 and np.array_equal(x, dumps[1][name]), name
    import bench
    key, vi, vf = bench.gen_groupby(200_000, 1000, 1)
    uk = np.unique(key)
    cnt = np.bincount(key)[uk]
    assert np.array_equal(d["groupby_key"], uk) and np.array_equal(d["groupby_len"], cnt)
    assert np.array_equal(d["groupby_sum"], np.bincount(key, weights=vi)[uk])
    assert np.allclose(d["groupby_mean"], np.bincount(key, weights=vf)[uk] / cnt, rtol=1e-12, atol=0)
    probe, build = bench.gen_join(200_000, 20_000, 2)
    assert np.array_equal(d["join_dense_left_idx"], np.arange(probe.size)) and np.array_equal(d["join_dense_right_idx"], np.argsort(build)[probe])


def test_dump_outputs_samples_long_outputs_under_64mb(tmp_path):
    """An output beyond its share of 64 MB is cut to rows at seeded positions (the same ones every time); nulls become NaN."""
    import bench
    n = 5_000_000
    outs = {"long": (np.arange(n, dtype=np.int64), np.arange(n) % 7 != 0), "short": (np.arange(5, dtype=np.uint32), None)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64_000_000
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a["short"].dtype == np.float64 and np.array_equal(a["short"], np.arange(5))
    got = a["long"]
    assert got.size < n and np.array_equal(got, b["long"], equal_nan=True)
    kept = got[~np.isnan(got)]
    assert np.all(np.diff(kept) > 0) and np.all(kept % 7 != 0) and 0 < np.isnan(got).sum() < got.size


@pytest.mark.gpu
def test_b200_arm_dumps_what_the_reference_arm_computes(tmp_path):
    """Both arms on the same seeded inputs: group keys, lengths, integer sums and join tuples exact, means within 1e-6 relative."""
    line = run_bench("--no-cpu-baseline", "--e2e-steps", "0", "--dump-outputs", str(tmp_path / "gpu"), impl="b200")
    assert line["steps"] == 1 and line["verified"]
    run_bench("--dump-outputs", str(tmp_path / "ref"))
    run_bench("--workload", "join", "--join-keys", "sparse", "--dump-outputs", str(tmp_path / "ref"))
    gpu, ref = _load(tmp_path / "gpu"), _load(tmp_path / "ref")
    assert sorted(gpu) == sorted(ref) == ["groupby_key", "groupby_len", "groupby_mean", "groupby_sum",
                                          "join_dense_left_idx", "join_dense_right_idx", "join_sparse_left_idx", "join_sparse_right_idx"]
    for name, x in gpu.items():
        if name == "groupby_mean":
            assert np.allclose(x, ref[name], rtol=1e-6, atol=0)
        else:
            assert np.array_equal(x, ref[name]), name

"""bench.py's output contract as far as it can be checked without a GPU: the reference arm (`--impl reference`, the
oracle port on the host cores) prints exactly one JSON line on stdout with the keys the driver reads, and under a
multi-rank launch only rank 0 prints."""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ensemble", "4",
           "--ref-pairs", "4000"]
    return subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    res = _run()
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert REQUIRED <= set(line)
    assert line["impl"] == "reference" and line["metric"] == "anchor_pairs_per_second" and line["unit"] == "anchor-pairs/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]
    assert "all-vs-all ensemble" in line["config"]["workload"] and line["scaling"] == "strong"   # the north-star workload is the default


def test_reference_arm_does_not_map_the_product_library():
    """The CPU arm must not load the CUDA library or the host extension (it only needs benchdata and the oracle)."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--ensemble', '3', "
            "'--ref-pairs', '2000']; runpy.run_path('bench.py', run_name='__main__'); "
            "maps = open('/proc/self/maps').read(); "
            "assert 'liblocohd_b200' not in maps and 'loco_hd.cpython' not in maps, 'product library mapped'; "
            "assert 'loco_hd_b200' not in sys.modules and 'loco_hd' not in sys.modules")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]


def test_reference_arm_other_ranks_stay_silent():
    res = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.strip() == ""


def test_sample_parity_helper():
    """bench.sample_parity (the GPU arm's check of every sampled job against the oracle) on a small ensemble, with the
    oracle's own results standing in for the GPU's: 0 for identical results, the injected error otherwise, nan (not an
    exception) when the results do not cover the sample."""
    import importlib.util

    import numpy as np

    import oracle

    spec = importlib.util.spec_from_file_location("_bench_mod", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    oracle.build()
    base = bench.synth.gen(9, 12, 8, 7)
    # a small stand-in workload with the structure of the default one: every pair of 4 members, every primitive an anchor
    clouds = [bench.synth.partner(base, 1.5, 3000 + i) for i in range(4)]
    groups = [(s, np.arange(base.n)) for s in range(4)]
    jobs = [(i, j) for i in range(4) for j in range(i + 1, 4)]
    wl = bench.Workload("cfg5", "test", 7, ("uniform", (3.0, 10.0)), clouds, groups, jobs, scaling="strong", means_only=True)
    op = bench.oracle_params(oracle, wl)
    ids = bench.sample_jobs(wl, 3 * base.n)
    assert ids == [0, 1, 2]
    got = []
    p, dt, steps, members = bench.oracle_run_jobs(oracle, op, wl, ids, n_threads=1, collect=got)
    assert p == 3 * base.n and len(got) == 3 and all(len(g) == base.n for g in got)
    means = np.array([g.mean() for g in got] + [0.0, 0.0, 0.0])
    assert bench.sample_parity(wl, ids, got, means, True) == 0.0
    means[2] += 1e-3
    assert abs(bench.sample_parity(wl, ids, got, means, True) - 1e-3) < 1e-12
    flat = np.concatenate(got)
    assert bench.sample_parity(wl, ids, got, flat, False) == 0.0
    flat[base.n + 5] += 2e-3
    assert abs(bench.sample_parity(wl, ids, got, flat, False) - 2e-3) < 1e-12
    assert np.isnan(bench.sample_parity(wl, ids, got, flat[: base.n], False))
    assert np.isnan(bench.sample_parity(wl, ids, got, means[:1], True))


def test_other_workload_entry_is_built_from_a_measurement(monkeypatch):
    """bench.other_workload (the `other_workloads` entries of the GPU arm's line) with the device measurement replaced
    by a canned result: the entry carries the keys the line documents."""
    import argparse
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("_bench_mod2", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    seen = {}

    def fake_measure(wl, ctx, local_rank, ranks, steps, warmup, args, clocks=True):
        seen.update(name=wl.name, steps=steps, warmup=warmup, clocks=clocks, solo=type(ranks).__name__)
        return {"value": 1.0e8, "step_ms": 2.0, "e2e": {"value": 9.0e7}, "launches": 12, "f_walk": 1.0e9, "f_gather": 1.0e8,
                "prof": {"score": (6.0, 3), "fill": (3.0, 3), "unused": (0.0, 0)}, "sizes": np.array([100, 200])}

    monkeypatch.setattr(bench, "measure", fake_measure)
    args = argparse.Namespace(steps=20, warmup=5, pairs=1, models=2, frames=2, ensemble=1000)
    out = bench.other_workload("cfg3", args, None, 0, 30.0)
    assert seen == {"name": "cfg3", "steps": 5, "warmup": 3, "clocks": False, "solo": "Solo"}
    assert out["value"] == 1.0e8 and out["anchor_pairs_per_step"] == 2 * 300 and out["gpu_launches"] == 12
    assert out["kernel_ms_per_step"] == {"score": 1.2, "fill": 0.6} and abs(sum(out["kernel_share"].values()) - 1.0) < 1e-12
    assert out["env_size_mean"] == 150.0 and out["roofline_step_frac_fp64"] > 0


def _load_bench(name):
    spec = importlib.util.spec_from_file_location(name, ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writes_float64_within_the_cap(tmp_path):
    """bench.dump_outputs (--dump-outputs): small results are written whole; above 64 MB in all the same seeded,
    sorted positions are kept on every run, and each rank of a multi-rank launch gets its share of the cap."""
    bench = _load_bench("_bench_mod3")
    small = np.arange(10, dtype=np.float64)
    p = bench.dump_outputs(tmp_path / "a", small, True, 0, 1)
    assert p == tmp_path / "a" / "job_means.npy" and np.array_equal(np.load(p), small)
    big = np.arange(bench.DUMP_BYTES // 8 + 1000, dtype=np.float64)   # value = position
    p1 = bench.dump_outputs(tmp_path / "b", big, False, 0, 1)
    p2 = bench.dump_outputs(tmp_path / "c", big, False, 0, 1)
    v1 = np.load(p1)
    assert p1.name == "scores_sample.npy" and v1.dtype == np.float64 and 0 < v1.nbytes <= bench.DUMP_BYTES
    assert np.all(np.diff(v1) > 0) and v1[-1] < len(big) and np.array_equal(v1, np.load(p2))
    p3 = bench.dump_outputs(tmp_path / "d", big, False, 1, 2)
    assert p3.name == "scores_rank1_sample.npy" and np.load(p3).nbytes <= bench.DUMP_BYTES // 2


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_steps_results(tmp_path, oracle_mod):
    """--dump-outputs on a 4-member ensemble: job_means.npy holds the 6 structure-pair means of the last timed step,
    which equal the oracle's within 1e-9."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "3", "--ensemble", "4",
           "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout)["steps"] == 2
    got = np.load(tmp_path / "job_means.npy")
    bench = _load_bench("_bench_mod4")
    wl = bench.make_workload("cfg5", 0, 1, argparse.Namespace(ensemble=4))
    op = bench.oracle_params(oracle_mod, wl)
    want = []
    for j in range(len(wl.jobs)):
        a, b, anchors = wl.job_arrays(j)
        want.append(oracle_mod.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, wl.threshold).mean())
    assert got.dtype == np.float64 and got.shape == (6,)
    assert np.abs(got - np.array(want)).max() <= 1e-9

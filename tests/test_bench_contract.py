"""bench.py's measurement contract, checked on CODE (not on committed artefacts): the host-side pieces on the CPU (the
reference arm, sharding of the C4 catalog, argument checks, the roofline bookkeeping constants) and, GPU-marked, one short
run of the real thing whose JSON line must carry every key the driver and the judge read."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H

sys.path.insert(0, H.ROOT)
import bench  # noqa: E402

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"}


def _run(*args, timeout=600):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    return subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, env=env)


def test_reference_arm_runs_on_the_host():
    out = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--objects", "2000")
    assert out.returncode == 0, out.stderr[-500:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["metric"] == "RSO UKF predict+update per second" and d["unit"] == "object-updates/s" and d["higher_is_better"] is True
    assert d["scaling"] == "strong" and d["config"]["workload"].startswith("C4") and d["warmup"] >= 1 and d["steps"] == 2


def test_gpus_flag_must_match_the_launch():
    out = _run("--gpus", "2", "--steps", "1")
    assert out.returncode != 0 and "torch.distributed.run" in (out.stderr + out.stdout)


def test_steps_and_dump_arguments_are_checked():
    out = _run("--steps", "0")
    assert out.returncode != 0 and "--steps must be at least 1" in out.stderr
    out = _run("--impl", "reference", "--dump-outputs", "unused")
    assert out.returncode != 0 and "--dump-outputs" in out.stderr


def test_c4_shards_are_slices_of_one_catalog():
    """Strong scaling: the job's inputs must not depend on the number of ranks."""
    from ssa_gym_b200.dist import shard_bounds
    total = 30011
    cat, x, P0, zn = bench.workload_inputs(total, 0, 2)
    assert cat.shape == (total, 6) and zn.shape == (2, total, 3)
    for world in (2, 3, 8):
        parts = [bench.workload_inputs(total, r, 2, *shard_bounds(total, world, r)) for r in range(world)]
        assert np.array_equal(np.concatenate([q[0] for q in parts]), cat)
        assert np.array_equal(np.concatenate([q[1] for q in parts]), x)
        assert np.array_equal(np.concatenate([q[3] for q in parts], axis=1), zn)


def test_catalog_layout_and_bookkeeping_constants():
    class A:
        workload, objects = "c4", 0
    tot = [bench.catalog_layout(A, 8, r) for r in range(8)]
    assert all(t[0] == 1_000_000 and t[4] == "strong" for t in tot) and tot[0][1] == 0 and tot[7][2] == 1_000_000
    assert sum(t[2] - t[1] for t in tot) == 1_000_000 and all(tot[r][2] == tot[r + 1][1] for r in range(7))
    A.workload = "c2"
    t = bench.catalog_layout(A, 4, 3)
    assert t[0] == 80000 and (t[1], t[2]) == (0, 20000) and t[4] == "weak"
    # SURVEY 8(d): 39 kflop and 920 B per object-step; the per-kernel split adds up
    assert bench.FLOP_PER_UNIT_REF == 39.0e3 and bench.BYTES_PER_UNIT_REF == 920
    assert abs(bench.FLOP_PREDICT_TILE_REF + bench.FLOP_UPDATE_TILE_REF + 2 * 0.32e3 - bench.FLOP_PER_UNIT_REF) < 0.5e3
    assert bench.BYTES_PER_UNIT == 698 and bench.FLOP_PER_UNIT < bench.FLOP_PER_UNIT_REF


@pytest.mark.gpu
def test_bench_line_carries_the_contract(tmp_path):
    out = _run("--steps", "3", "--warmup", "3", "--objects", "60000", "--cpu-seconds", "1", "--dump-outputs", str(tmp_path), timeout=900)
    assert out.returncode == 0, out.stderr[-800:]
    dump = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    shapes = {"x_true": (60000, 6), "x_filter": (60000, 6), "P_filter": (60000, 6, 6), "obs": (60000, 12), "delta_pos": (60000,),
              "delta_vel": (60000,), "sigma_pos": (60000,), "sigma_vel": (60000,), "trace": (60000,), "status": (60000,),
              "inflations": (60000,), "catalog_stats": (1, 5)}
    assert {k: v.shape for k, v in dump.items()} == shapes and all(v.dtype == np.float64 for v in dump.values())
    assert np.isfinite(dump["x_filter"]).all() and dump["catalog_stats"][0, 2] == 60000
    assert dump["catalog_stats"][0, 0] == dump["delta_pos"].max()
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert BASE_KEYS | {"cpu_baseline"} <= set(d), BASE_KEYS - set(d)
    assert d["unit"] == "object-updates/s" and d["higher_is_better"] is True and d["scaling"] == "strong" and d["dtype"] == "f64"
    assert d["vs_baseline"] is None and d["config"]["workload"].startswith("C4") and "l2" in d["config"]
    assert d["warmup"] >= 3 and d["steps"] == 3 and d["n_gpus"] == 1
    assert abs(d["value"] - d["config"]["objects_total"] / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "whole_step"} <= set(r) and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert 0 < r["frac"] < 1 and r["kernel"] == "k_predict_tile"
    assert abs(r["achieved"] - bench.FLOP_PREDICT_TILE_REF * 60000 / (r["kernel_ms"] * 1e-3) / 1e12) < 1e-9 * r["achieved"]
    assert r["whole_step"]["algorithmic_bytes"] == 920 * 60000 and 0 < r["whole_step"]["frac"] < 1
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e) and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert e["value"] != d["value"]                       # measured separately, not a copy of the device-timed value
    c = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] == "port" and c["cores"] >= 1
    assert c["reference_style_python"]["single_process"]["value"] > 0
    g = d["extra"]["c4_reward_gather"]
    assert g["gathered_ranks"] == 1 and g["objects_gathered"] == 60000 and g["in_timed_events"] is True
    assert d["gpu_launches"] >= 6 * d["steps"]            # 4 UKF kernels + 2 reward-reduction kernels per step
    assert d["extra"]["c2"]["value"] > 0 and d["extra"]["c3"]["value"] > 0
    k = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(k)

"""bench.py's output contract (the driver parses ONE JSON line from stdout).

CPU: the reference arm (`--impl reference`, the oracle port on the host cores) runs here and must print exactly one
line with the keys the driver reads.  GPU: the same for the default arm, plus the tier-specific objects (roofline,
cpu_baseline, e2e, clocks, gpu_launches).
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def _run(*args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=600, env={**os.environ, **(env or {})})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, f"stdout must carry exactly one line, got {len(lines)}: {r.stdout[:500]}"
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line(tmp_path):
    d = _run("--impl", "reference", "--steps", "5", "--warmup", "3", "--dump-outputs", str(tmp_path))
    assert d["impl"] == "reference"
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["metric"] == "rollout_steps_per_sec" and d["unit"] == "rollout-steps/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] == "omni_1000x56" and "model" not in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["vs_baseline"] is None
    assert d["steps"] == 5
    # --dump-outputs: the last timed optimize() as the caller received it
    assert sorted(os.listdir(tmp_path)) == [f"omni_1000x56.{n}.npy" for n in sorted(
        ("vx", "vy", "wz", "fail_flag", "furthest_reached_path_point"))]
    for name in ("vx", "vy", "wz"):
        a = np.load(tmp_path / f"omni_1000x56.{name}.npy")
        assert a.dtype == np.float32 and a.shape == (56,) and np.isfinite(a).all(), name
    assert np.abs(np.load(tmp_path / "omni_1000x56.vx.npy")).max() > 1e-3
    assert np.load(tmp_path / "omni_1000x56.fail_flag.npy").tolist() == [0.0]
    # the same oracle build through 3 warmup + 5 timed cycles
    import bench
    sc, noise_kind = bench.pick_scenario("omni_1000x56", 0, 1)
    e = bench.oracle_engine(sc, noise_kind)
    results = [e.optimize(sc.cycle) for _ in range(3 + 5)]
    e.close()
    _assert_dump_is_last(tmp_path, "omni_1000x56", results)


def _assert_dump_is_last(directory, workload, results):
    """the dump of `workload` is the last of `results` bit for bit, and the step before it differs"""
    last, before = results[-1], results[-2]
    for name in ("vx", "vy", "wz"):
        np.testing.assert_array_equal(np.load(directory / f"{workload}.{name}.npy"), getattr(last, name), err_msg=name)
    assert any(not np.array_equal(getattr(last, n), getattr(before, n)) for n in ("vx", "vy", "wz"))
    assert np.load(directory / f"{workload}.fail_flag.npy").tolist() == [float(last.fail_flag)]
    f = last.furthest_reached_path_point
    assert np.load(directory / f"{workload}.furthest_reached_path_point.npy").tolist() == [-1.0 if f is None else float(f)]


def test_reference_arm_takes_steps_and_warmup_as_given():
    """only the defaults of the reference arm are bounded by time: an explicit --warmup 8 on configs[3] (~1.6 s a cycle on one
    core) runs 8 warmup cycles, not the 7 that fit in 20 s"""
    d = _run("--impl", "reference", "--workload", "sharded_262144x100", "--steps", "1", "--warmup", "8")
    assert d["steps"] == 1 and d["warmup"] == 8


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr, r.stderr


def test_reference_arm_other_ranks_stay_silent():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2"],
                       capture_output=True, text=True, timeout=300, env={**os.environ, "RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_default_arm_line_on_the_gpu(tmp_path, product_fns):
    d = _run("--steps", "60", "--warmup", "3", "--dump-outputs", str(tmp_path / "full"))
    assert BASE_KEYS | {"roofline", "cpu_baseline", "clocks", "gpu_launches", "latency_ms"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 60 and d["dtype"] == "f32" and d["scaling"] == "weak"
    assert d["config"]["workload"] == "omni_1000x56"
    roof = d["roofline"]
    assert roof["bound"] in ("hbm", "issue") and 0 < roof["frac"] < 1
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert d["gpu_launches"] == 60                      # one fused kernel per optimize()
    assert d["e2e"]["h2d_bytes_per_step"] > 10000 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] < d["value"]               # end to end includes the copies and the host
    assert d["cpu_baseline"]["value"] < d["e2e"]["value"]
    assert d["latency_ms"]["e2e_p50"] < 0.3             # north_star: 1000 x 56 under 0.3 ms per optimize()
    # the other BASELINE configs ride in the same line, measured in the same process, each with its in-run oracle check
    for name in ("obstacles_16384x56", "obstacles_dense_16384x56", "sharded_262144x100", "robots_256"):
        rec = d[name]
        assert "error" not in rec, rec
        assert rec["ms_per_step"] > 0 and rec["e2e"]["value"] > 0 and "roofline" in rec and "cpu_baseline" in rec
        assert rec["parity"]["status"] == "ok", rec["parity"]
        assert rec["steps"] == 60 and rec["warmup"] == 3, name   # --steps / --warmup hold for the nested records too
    # SURVEY 8d: the footprint-branch fraction of config 3, counted by the CPU oracle of the same run
    dense = d["obstacles_dense_16384x56"]["cpu_baseline"]["footprint_branch"]
    warm = [v for k, v in dense.items() if k.startswith("cycle_")][0]["ObstaclesCritic"]
    assert warm["fraction_of_visited"] > 0.08
    assert "first_cycle_zero_control_sequence" in d["obstacles_16384x56"]["cpu_baseline"]["footprint_branch"]
    # --dump-outputs: what the last timed step returned, for every workload of the line
    shapes = {"omni_1000x56": (56,), "obstacles_16384x56": (56,), "obstacles_dense_16384x56": (56,),
              "sharded_262144x100": (100,), "robots_256": (256, 56)}
    for wl, shape in shapes.items():
        for name in ("vx", "vy", "wz"):
            a = np.load(tmp_path / "full" / f"{wl}.{name}.npy")
            assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all(), (wl, name)
        for name in ("fail_flag", "furthest_reached_path_point"):
            a = np.load(tmp_path / "full" / f"{wl}.{name}.npy")
            assert a.dtype == np.float64 and a.shape == (shape[:-1] or (1,)), (wl, name)
    assert np.abs(np.load(tmp_path / "full" / "omni_1000x56.vx.npy")).max() > 1e-3
    # the dump is the LAST timed step: the same resident cycles, 3 warmup + 60 timed, replayed here give it bit for bit
    import bench
    from mpcholonavigation_b200 import Engine
    sc, _ = bench.pick_scenario("omni_1000x56", 0, 1)
    e = Engine(product_fns, **dict(sc.cfg, device=0, seed=3))
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*sc.noise())
    e.upload_cycle(sc.cycle)
    results = [e.optimize_resident() for _ in range(3 + 60)]
    e.close()
    _assert_dump_is_last(tmp_path / "full", "omni_1000x56", results)


def test_reference_arm_prints_the_same_config_object():
    """same_config / warmup_match of the driver: the reference arm echoes the GPU arm's config and honours --warmup"""
    import bench
    from mpcholonavigation_b200 import scenarios
    sc = scenarios.config1()
    want = bench.make_config("omni_1000x56", sc, "injected", 1, "peer", True)
    d = _run("--impl", "reference", "--steps", "3", "--warmup", "7")
    assert d["config"] == want and d["warmup"] == 7


@pytest.mark.parametrize("n", [256, 128, 32])
def test_robots_roofline_from_the_committed_counters(n):
    """robots_256.roofline at N = 1, 2, 8: traffic and the issue side come from the counters of one 256-robot step, scaled to
    the rank's robots; the reported bound is the larger fraction and frac == achieved / peak"""
    import bench
    peaks = bench.load_peaks()
    kc = bench.kernel_counters("robots_step", 2000, 56)
    assert kc and kc["n_robots"] == 256 and kc["launches"] == 4
    step_ms = 0.5 * n / 256 + 0.1
    alg = n * bench.algorithmic_bytes(2000, 56, 40, 10000)
    roof = bench.make_roofline("robots", step_ms, alg, n * 2000, 56, peaks, "note")
    roof = bench.robots_roofline(roof, kc, n, step_ms, peaks)
    assert roof["traffic"] == int(kc["dram_bytes"] * n / 256) and roof["traffic"] > alg
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12
    other = roof.get("hbm") or roof.get("issue")
    assert other and other["frac"] <= roof["frac"] and {other["bound"], roof["bound"]} == {"hbm", "issue"}
    assert abs(sum(v["share_of_ncu_time"] for v in roof["per_kernel_ncu"].values()) - 1.0) < 1e-9
    assert bench.robots_roofline({"frac": 0.1}, None, n, step_ms, peaks) == {"frac": 0.1}

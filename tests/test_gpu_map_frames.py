"""Parity of the CUDA paths against the CPU oracle on costmaps away from the world origin (tests/map_frames.py): offset and
negative origins up to 1e5 m, non-square windows, resolutions 0.01 - 0.1 m, poses on cell edges and corners, Nav2's
rolling window, and robot groups whose members all see different frames.

Bars as in test_gpu_parity.py: cell indices and trajectories bit-exact; per-critic and total costs within rtol 1e-4,
atol 5e-6; controls within rtol 1e-4, atol 1e-6; fail flag and furthest point equal.  Every test also checks the device's
cells against cells_fp64 (numpy worldToMap) of the device's own trajectories, and asserts that it reached what it is
about (poses whose fp32 cell is not their fp64 cell, both sides of the edges, off-map cells), so that a change that makes
a scenario miss its edge cases fails instead of passing vacuously.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from mpcholonavigation_b200 import Engine, abi, optimize_group_device, optimize_sharded, scenarios, sharding
from mpcholonavigation_b200.api import Cycle, circle_footprint, make_robot
from tests import map_frames as mf
from tests.test_gpu_group_device_inputs import _host_batch, _inputs, _same

pytestmark = pytest.mark.gpu

RTOL, COST_ATOL = 1e-4, 5e-6
# controls: 1e-6 in test_gpu_parity.py; the 401 x 263 window's scene puts 2e-6 between the fp32 softmax sums of the two
# sides on every path alike (cells, trajectories and costs meeting their bars), so the absolute floor here is 3e-6
ATOL = 3e-6
FRAMES = list(mf.FRAMES)
RECT = np.array([[0.25, 0.15], [-0.25, 0.15], [-0.25, -0.15], [0.25, -0.15]])


def _circle_robot():
    return make_robot(circle_footprint(0.25), inscribed_radius=0.25, circumscribed_radius=0.25, inflation_layer_found=True,
                      inflation_cost_scaling_factor=3.0, track_unknown=False)


def _rect_robot():
    return make_robot(RECT, inscribed_radius=0.15, circumscribed_radius=float(np.hypot(0.25, 0.15)),
                      inflation_layer_found=True, inflation_cost_scaling_factor=3.0, track_unknown=False)


def _omni(frame, batch=1000, steps=56, seed=3, edge_margin=0.1):
    """config1-like: the default Omni critic set on the frame's world, the robot near the window's edge"""
    wd = mf.world(frame, seed, edge_margin=edge_margin)
    return wd, scenarios.Scenario("omni_" + frame.name, scenarios._omni_cfg(batch, steps),
                                  scenarios.omni_default_critics(True), _circle_robot(), wd.cycle(), 1)


def _obstacles(frame, dense, batch=2048, steps=56, seed=5):
    """config3-like: ObstaclesCritic alone in footprint mode; dense: a rectangular robot boxed in by a ring of discs"""
    wd = mf.world(frame, seed, ring=0.47 if dense else None, inscribed_radius=0.15 if dense else 0.25, edge_margin=0.1)
    critics = [("ObstaclesCritic", dict(consider_footprint=1, inflation_radius=0.55, cost_scaling_factor=3.0))]
    return wd, scenarios.Scenario("obstacles_" + frame.name, scenarios._omni_cfg(batch, steps), critics,
                                  _rect_robot() if dense else _circle_robot(), wd.cycle(), 3)


def _engine(fns, sc, noise=None, outputs=True, device_map=False, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*(sc.noise() if noise is None else noise))
    if outputs:
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    if device_map:
        e.set_costmap_residency(True)
    return e


def _on_device(cycle):
    return dataclasses.replace(cycle, costmap=torch.from_numpy(np.ascontiguousarray(cycle.costmap)).cuda())


def _own_cells(g, frame, label):
    """the device's cells are cells_fp64 of the device's own trajectories"""
    x, y, _ = g.get_trajectories()
    want = mf.cells_fp64(x, y, frame)
    got = g.get_cells()
    bad = np.flatnonzero(got.ravel() != want.ravel())
    if bad.size:
        i = bad[0]
        xf, yf = x.ravel()[i], y.ravel()[i]
        q = ((float(xf) - frame.origin[0]) / frame.resolution, (float(yf) - frame.origin[1]) / frame.resolution)
        raise AssertionError(f"{label}: {bad.size} cells differ from cells_fp64; first pose ({xf!r}, {yf!r}) fp64 "
                             f"quotients {q}, device {got.ravel()[i]}, fp64 {want.ravel()[i]}, frame {frame}")
    return want


def _critic_rows(g, o, n_critics, label):
    """per-critic costs within rtol 1e-4, atol 5e-6 - or one ulp of the trajectory's fp32 total, whichever is larger:
    the oracle records a critic's row as the difference of the running fp32 total around it, so with totals above 64
    (collisions, a second iteration's accumulated costs) its rows are quantised to that ulp"""
    floor = np.maximum(COST_ATOL, np.spacing(np.abs(o.get_costs())))
    for q in range(n_critics):
        a, b = g.get_critic_costs(q), o.get_critic_costs(q)
        bad = np.abs(a - b) > floor + RTOL * np.abs(b)
        assert not bad.any(), f"{label}: critic {q}: {bad.sum()} rows, first {np.flatnonzero(bad)[:4]} {a[bad][:4]} vs {b[bad][:4]}"


def _bars(g, o, rg, ro, n_critics, label, outputs=True, control_atol=ATOL):
    if outputs:
        assert np.array_equal(g.get_cells(), o.get_cells()), f"{label}: {np.count_nonzero(g.get_cells() != o.get_cells())} cells"
        for name, a, b in zip("x y yaw".split(), g.get_trajectories(), o.get_trajectories()):
            assert np.array_equal(a, b), f"{label}: trajectory {name} differs in {np.count_nonzero(a != b)} places"
        _critic_rows(g, o, n_critics, label)
    np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=COST_ATOL, err_msg=f"{label}: total costs")
    for name in ("vx", "vy", "wz"):
        np.testing.assert_allclose(getattr(rg, name), getattr(ro, name), rtol=RTOL, atol=control_atol,
                                   err_msg=f"{label}: control {name}")
    assert rg.fail_flag == ro.fail_flag, label
    assert rg.furthest_reached_path_point == ro.furthest_reached_path_point, label


def _set_env(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _clear_env(monkeypatch, env):
    for k in env:
        monkeypatch.delenv(k, raising=False)


# ------------------------------------------------------------------------------------------------
# A. the cell index itself: injected trajectories on cell edges through the tile kernel (score mode)
# ------------------------------------------------------------------------------------------------
# poses whose fp32 cell differs from the fp64 cell, at least, among edge_poses.  res_003 and res_01 have fewer by the
# arithmetic of their grids: at 0.1 m the fp64 edges sit at five fixed fractions of an fp32 ulp and fl32(origin) moves
# them onto pose values, never across one; at 0.03 m most fp32 edges fall between the same two poses as the fp64 edge.
MIN_FP32_DIFF = {"res_003": 30, "res_01": 0}
CRITIC_SETS = {
    "cost_footprint_obstacles": [("CostCritic", dict(consider_footprint=1, cost_weight=3.81, critical_cost=300.0,
                                                     collision_cost=1000000.0, near_goal_distance=0.5)),
                                 ("ObstaclesCritic", dict(consider_footprint=1, inflation_radius=0.55, cost_scaling_factor=3.0,
                                                          near_goal_distance=0.5))],
    "cost_point": [("CostCritic", dict(consider_footprint=0, cost_weight=3.81, critical_cost=300.0, collision_cost=1000000.0,
                                       near_goal_distance=0.5, trajectory_point_step=1))],
}


def _painted(frame):
    """every cell differs from its four neighbours; the window's border ring is inscribed (253), so that the footprint
    branch runs next to the edges with vertices off the map"""
    yy, xx = np.mgrid[0:frame.size_y, 0:frame.size_x]
    cm = ((xx * 37 + yy * 101) % 97 + 10).astype(np.uint8)
    cm[0, :] = cm[-1, :] = cm[:, 0] = cm[:, -1] = scenarios.INSCRIBED
    return cm


@pytest.mark.parametrize("critics", list(CRITIC_SETS))
@pytest.mark.parametrize("frame", FRAMES)
def test_edge_poses_cells_and_costs(product_fns, oracle_fns, frame, critics):
    f = mf.FRAMES[frame]
    p = mf.edge_poses(f)
    T = 56
    B = p.x.size // T
    x, y = p.x.reshape(B, T), p.y.reshape(B, T)
    yaw = np.random.default_rng(1).uniform(-np.pi, np.pi, (B, T)).astype(np.float32)
    zeros = np.zeros((B, T), np.float32)
    cx, cy = f.centre
    px, py, pyaw = scenarios.straight_path(cx, cy, 0.3, 40, 0.05)
    cyc = Cycle(pose=(cx, cy, 0.3), goal=(cx + 50.0, cy + 50.0), path_x=px, path_y=py, path_yaw=pyaw,
                   costmap=_painted(f), resolution=f.resolution, origin=f.origin)
    cfg = scenarios._omni_cfg(B, T)
    res = []
    for fns in (product_fns, oracle_fns):
        e = Engine(fns, **cfg)
        e.set_robot(_rect_robot())
        e.set_critics(CRITIC_SETS[critics])
        e.set_outputs(cells=True, critic_costs=True)
        res.append((e, e.score_trajectories(cyc, zeros, zeros, zeros, x, y, yaw)))
    (g, (cg, fg, failg)), (o, (co, fo, failo)) = res
    want = mf.cells_fp64(x, y, f)
    got = g.get_cells()
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, (f"{bad.size} cells differ; first pose ({x.ravel()[bad[0]]!r}, {y.ravel()[bad[0]]!r}) kind "
                           f"{mf.KINDS[p.kind[bad[0]]]}: device {got.ravel()[bad[0]]}, fp64 {want.ravel()[bad[0]]}")
    cm = abi.Costmap()
    cm.size_x, cm.size_y, cm.resolution = f.size_x, f.size_y, f.resolution
    cm.origin_x, cm.origin_y = f.origin
    w2m = oracle_fns["world_to_map"]
    sel = np.flatnonzero(p.kind != mf.KINDS.index("random"))   # the oracle's worldToMap on every edge and off-map pose
    oc = np.array([w2m(C.byref(cm), float(p.x[i]), float(p.y[i])) for i in sel], np.int32)
    assert np.array_equal(oc, want.ravel()[sel])
    _critic_rows(g, o, len(CRITIC_SETS[critics]), frame)
    np.testing.assert_allclose(cg, co, rtol=RTOL, atol=COST_ATOL)
    assert failg == failo and fg == fo
    # coverage
    cand, sure = mf.filter_fp32(p.x, p.y, f)
    assert np.count_nonzero(cand != want.ravel()) >= MIN_FP32_DIFF.get(frame, 100)
    for key, (below, above) in mf.edge_sides(p, f).items():
        assert below > 0 and above > 0, key
    if frame == "filter_off":
        assert not sure.any()
    assert (want == -1).any() and (o.get_critic_costs(0) > 0).any()
    g.close(); o.close()


# ------------------------------------------------------------------------------------------------
# B. the robot on a cell corner through optimize(): every rollout path's cell mapping, within ulps of the corner
# ------------------------------------------------------------------------------------------------
CORNER_PATHS = {"fused_exact": ({}, False), "fused_outputs": ({}, True), "two_kernel": ({"MPPI_FUSED": "0"}, True),
                "stream": ({"MPPI_STREAM_MIN_BATCH": "1"}, True)}


def _corner_scenario(frame, corner):
    k = {"interior": (frame.size_x // 2, frame.size_y // 3), "origin": (0, 0), "far": (frame.size_x, frame.size_y)}[corner]
    pose = (*mf.grid_point(frame, *k), 0.0)
    cm = np.zeros((frame.size_y, frame.size_x), np.uint8)
    for (dx, dy), c in zip(((-1, -1), (0, -1), (-1, 0), (0, 0)), (40, 80, 120, 160)):
        if 0 <= k[0] + dx < frame.size_x and 0 <= k[1] + dy < frame.size_y:
            cm[k[1] + dy, k[0] + dx] = c
    px, py, pyaw = scenarios.straight_path(pose[0], pose[1], 0.0, 40, 0.05)
    cyc = Cycle(pose=pose, goal=(float(px[-1]), float(py[-1])), goal_checker_xy_tolerance=0.25, path_x=px, path_y=py,
                   path_yaw=pyaw, costmap=cm, resolution=frame.resolution, origin=frame.origin)
    cfg = scenarios._omni_cfg(1000, 56, vx_std=5e-4, vy_std=5e-4)
    sc = scenarios.Scenario("corner", cfg, scenarios.omni_default_critics(True), _circle_robot(), cyc, 0)
    rng = np.random.default_rng(17)
    noise = (rng.standard_normal((1000, 56)).astype(np.float32) * np.float32(5e-4),
             rng.standard_normal((1000, 56)).astype(np.float32) * np.float32(5e-4), np.zeros((1000, 56), np.float32))
    return sc, noise, k


@pytest.mark.parametrize("path", list(CORNER_PATHS))
@pytest.mark.parametrize("corner", ["interior", "origin", "far"])
@pytest.mark.parametrize("frame", ["res_007_tall", "campus"])
def test_robot_on_a_cell_corner(product_fns, oracle_fns, monkeypatch, frame, corner, path):
    f = mf.FRAMES[frame]
    sc, noise, k = _corner_scenario(f, corner)
    env, outputs = CORNER_PATHS[path]
    _set_env(monkeypatch, env)
    g = _engine(product_fns, sc, noise, outputs=outputs)
    _clear_env(monkeypatch, env)
    o = _engine(oracle_fns, sc, noise)
    zero = np.zeros(56, np.float32)
    quadrants, diff = np.zeros(4, int), 0
    for cycle in range(3):
        for e in (g, o):
            e.set_control_sequence(zero, zero, zero)
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _bars(g, o, rg, ro, len(sc.critics), f"{path} cycle {cycle}", outputs=outputs)
        if outputs:
            _own_cells(g, f, f"{path} cycle {cycle}")
        x, y, _ = o.get_trajectories()
        mx = mf.axis_cells_fp64(x, f.origin[0], f.resolution, f.size_x) >= k[0]
        my = mf.axis_cells_fp64(y, f.origin[1], f.resolution, f.size_y) >= k[1]
        quadrants += np.bincount((mx * 1 + my * 2).ravel(), minlength=4)
        cand, _ = mf.filter_fp32(x, y, f)
        diff += np.count_nonzero(cand != mf.cells_fp64(x, y, f))
    assert (quadrants > 0).all(), quadrants
    assert diff > 0
    g.close(); o.close()


# ------------------------------------------------------------------------------------------------
# C. end-to-end parity per frame and per path
# ------------------------------------------------------------------------------------------------
PATHS = ["fused", "two_kernel", "copy_engine", "stream", "iteration_count_2", "eval_control_shift", "device_map", "sharded"]
ENV = {"two_kernel": {"MPPI_FUSED": "0"}, "copy_engine": {"MPPI_ZERO_COPY": "0"}, "stream": {"MPPI_STREAM_MIN_BATCH": "1"}}


def _coverage(wd, cells_seen, critic_seen):
    assert (cells_seen == -1).any(), "no rollout pose off the map"
    assert (mf.cells_fp64(wd.path_x, wd.path_y, wd.frame) == -1).any(), "every path point on the map"
    assert critic_seen, "CostCritic / ObstaclesCritic zero everywhere"


def _critic_seen(o, sc):
    return any((o.get_critic_costs(q) > 0).any() for q, (name, _) in enumerate(sc.critics)
               if name in ("CostCritic", "ObstaclesCritic"))


def _parity(product_fns, oracle_fns, monkeypatch, wd, sc, path, cycles=3):
    f = wd.frame
    noise = sc.noise()
    n_critics = len(sc.critics)
    cells_seen, critic_seen = [], False
    if path == "sharded":
        B = sc.cfg["batch_size"]
        shards = []
        for r in range(2):
            b0, b1 = sharding.shard_bounds(B, r, 2)
            e = Engine(product_fns, **dict(sc.cfg, batch_size=b1 - b0, shard_offset=b0, shard_total=B))
            e.set_robot(sc.robot)
            e.set_critics(sc.critics)
            e.set_noise(*[a[b0:b1] for a in noise])
            shards.append(e)
        o = _engine(oracle_fns, sc, noise)
        for cycle in range(cycles):
            rs, ro = optimize_sharded(shards, sc.cycle), o.optimize(sc.cycle)
            for name in ("vx", "vy", "wz"):
                np.testing.assert_allclose(getattr(rs, name), getattr(ro, name), rtol=RTOL, atol=ATOL, err_msg=name)
            assert rs.fail_flag == ro.fail_flag and rs.furthest_reached_path_point == ro.furthest_reached_path_point
            np.testing.assert_allclose(np.concatenate([e.get_costs() for e in shards]), o.get_costs(), rtol=RTOL, atol=COST_ATOL)
            cells_seen.append(o.get_cells())
            critic_seen |= _critic_seen(o, sc)
            for e in shards:
                e.set_control_sequence(ro.vx, ro.vy, ro.wz)
        _coverage(wd, np.concatenate(cells_seen), critic_seen)
        for e in shards + [o]:
            e.close()
        return
    env = ENV.get(path, {})
    _set_env(monkeypatch, env)
    kw = dict(iteration_count=2) if path == "iteration_count_2" else {}
    g = _engine(product_fns, sc, noise, **kw)
    _clear_env(monkeypatch, env)
    o = _engine(oracle_fns, sc, noise, **kw)
    d = _engine(product_fns, sc, noise, device_map=True) if path == "device_map" else None
    g1 = _engine(product_fns, sc, noise) if path == "iteration_count_2" else None
    dev_cycle = _on_device(sc.cycle) if d else None
    hist = np.arange(12, dtype=np.float32).reshape(4, 3) * 0.01
    if path == "eval_control_shift":
        g.set_control_history(hist)
        o.set_control_history(hist)
    for cycle in range(cycles):
        label = f"{f.name} {path} cycle {cycle}"
        if g1 is not None:
            # the oracle's second iteration starts from the device's first update: the second rollout is bit-comparable
            g1.set_control_sequence(*g.get_control_sequence())
            r1 = g1.optimize(sc.cycle)
            pin = [np.ascontiguousarray(a, dtype=np.float32) for a in (r1.vx, r1.vy, r1.wz)]
            f32p = oracle_fns["_lib"].oracle_set_iteration_controls.argtypes[2]
            assert oracle_fns["set_iteration_controls"](o.h, 0, *[a.ctypes.data_as(f32p) for a in pin]) == 0
        if path == "eval_control_shift":
            cmd_g, rg = g.eval_control(sc.cycle, True)
            cmd_o, ro = o.eval_control(sc.cycle, True)
            np.testing.assert_allclose(cmd_g, cmd_o, rtol=RTOL, atol=ATOL, err_msg=f"{label}: command")
            np.testing.assert_allclose(g.get_control_history(), o.get_control_history(), rtol=RTOL, atol=ATOL)
            np.testing.assert_allclose(np.stack(g.get_control_sequence()), np.stack(o.get_control_sequence()), rtol=RTOL, atol=ATOL)
        else:
            rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        # iteration_count 2 softmaxes the accumulated costs of both iterations (quirk R20), totals in the hundreds near
        # the window's edge: the controls get test_gpu_parity.test_iteration_count_two's 1e-5 floor
        _bars(g, o, rg, ro, n_critics, label, control_atol=1e-5 if g1 is not None else ATOL)
        _own_cells(g, f, label)
        if d is not None:
            rd = d.optimize(dev_cycle)
            for name in ("vx", "vy", "wz"):
                assert np.array_equal(getattr(rd, name), getattr(rg, name)), f"{label}: device map {name}"
            assert np.array_equal(d.get_cells(), g.get_cells()) and np.array_equal(d.get_costs(), g.get_costs()), label
            assert rd.fail_flag == rg.fail_flag and rd.furthest_reached_path_point == rg.furthest_reached_path_point
        cells_seen.append(o.get_cells())
        critic_seen |= _critic_seen(o, sc) or (g1 is not None and _critic_seen(g1, sc))
        # keep both sides on the same warm start so that the comparison stays point-wise
        for e in (g, d):
            if e is not None:
                e.set_control_sequence(*o.get_control_sequence())
        if path == "eval_control_shift":
            g.set_control_history(o.get_control_history())
    _coverage(wd, np.concatenate(cells_seen), critic_seen)
    for e in (g, o, d, g1):
        if e is not None:
            e.close()


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("frame", FRAMES)
def test_omni_parity(product_fns, oracle_fns, monkeypatch, frame, path):
    wd, sc = _omni(mf.FRAMES[frame])
    _parity(product_fns, oracle_fns, monkeypatch, wd, sc, path)


@pytest.mark.parametrize("path", ["fused", "stream"])
@pytest.mark.parametrize("dense", [False, True], ids=["plain", "dense"])
@pytest.mark.parametrize("frame", FRAMES)
def test_obstacles_footprint_parity(product_fns, oracle_fns, monkeypatch, frame, dense, path):
    wd, sc = _obstacles(mf.FRAMES[frame], dense)
    _parity(product_fns, oracle_fns, monkeypatch, wd, sc, path, cycles=2)


# ------------------------------------------------------------------------------------------------
# D. the rolling window in closed loop
# ------------------------------------------------------------------------------------------------
def _advance(pose, cmd, dt):
    x, y, yaw = pose
    c, s = np.cos(yaw), np.sin(yaw)
    vx, vy, wz = (float(v) for v in cmd)
    return (x + (vx * c - vy * s) * dt, y + (vx * s + vy * c) * dt, yaw + wz * dt)


@pytest.mark.parametrize("frame", ["odom", "campus"])
def test_rolling_window_closed_loop(product_fns, oracle_fns, monkeypatch, frame):
    """30 cycles of evalControl: the robot moves by the command, the window snaps to it (the origin moves by whole cells),
    the path is pruned behind the robot.  Fused host map, device map and stream layout against the oracle every cycle."""
    wd, sc = _omni(mf.FRAMES[frame], edge_margin=None)
    noise = sc.noise()
    fused = _engine(product_fns, sc, noise)
    dev = _engine(product_fns, sc, noise, device_map=True)
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1")
    stream = _engine(product_fns, sc, noise)
    monkeypatch.delenv("MPPI_STREAM_MIN_BATCH")
    o = _engine(oracle_fns, sc, noise)
    pose, speed = wd.pose, (0.0, 0.0, 0.0)
    origins, path_off_map = set(), False
    for cycle in range(30):
        cyc = wd.cycle(speed)
        cmd_o, ro = o.eval_control(cyc, True)
        for name, e, c in (("fused", fused, cyc), ("device map", dev, _on_device(cyc)), ("stream", stream, cyc)):
            label = f"{frame} cycle {cycle} {name}"
            cmd, r = e.eval_control(c, True)
            np.testing.assert_allclose(cmd, cmd_o, rtol=RTOL, atol=ATOL, err_msg=f"{label}: command")
            _bars(e, o, r, ro, len(sc.critics), label)
            _own_cells(e, wd.frame, label)
            e.set_control_sequence(*o.get_control_sequence())
            e.set_control_history(o.get_control_history())
        path_off_map |= bool((mf.cells_fp64(wd.path_x, wd.path_y, wd.frame) == -1).any())
        origins.add(wd.frame.origin)
        pose = _advance(pose, cmd_o, sc.cfg["model_dt"])
        speed = tuple(float(v) for v in cmd_o)
        wd = mf.prune_path(mf.rolling(wd, pose), pose)
    assert len(origins) >= 5, "the window never moved"
    assert path_off_map
    for e in (fused, dev, stream, o):
        e.close()


# ------------------------------------------------------------------------------------------------
# E. robot groups whose members see different frames
# ------------------------------------------------------------------------------------------------
def _bind(fns, engines):
    hs = (abi.H * len(engines))(*[e.h for e in engines])
    assert fns["batch_bind"](hs, len(engines)) == 0, fns["last_error"](engines[0].h)
    return hs


def _member_worlds(n):
    """member i: FRAMES entry i % 8, the robot of every even member 0.1 m from the window's edge, the windows of members
    8 - 15, 24 - 31, ... moved by a rolling step of their own"""
    out = []
    for i in range(n):
        f = mf.FRAMES[FRAMES[i % len(FRAMES)]]
        wd = mf.world(f, seed=100 + i, edge_margin=0.1 if i % 2 == 0 else None)
        if (i // len(FRAMES)) % 2 == 1:
            x, y, yaw = wd.pose
            step = (i % 5 + 1) * 1.37 * f.resolution
            wd = mf.rolling(wd, (x + step, y - step, yaw))
        out.append(wd)
    return out


def test_group_of_seventy_frames(product_fns, oracle_fns):
    """70 members (two chunks), origins, resolutions and window shapes all different within each launch, a third of them
    with device maps: mppi_optimize_batch and mppi_optimize_batch_resident against each member's oracle"""
    n, T = 70, 56
    wds = _member_worlds(n)
    scs = [scenarios.Scenario(f"m{i}", scenarios._omni_cfg(256, T), scenarios.omni_default_critics(True), _circle_robot(),
                              wd.cycle(), 1000 + i) for i, wd in enumerate(wds)]
    device = [i % 3 == 1 for i in range(n)]
    cycles = [_on_device(sc.cycle) if device[i] else sc.cycle for i, sc in enumerate(scs)]
    es = [_engine(product_fns, sc, device_map=device[i]) for i, sc in enumerate(scs)]
    for e, c in zip(es, cycles):
        e.upload_cycle(c)   # the members' staging fits their maps before the group's slices are bound
    hs = _bind(product_fns, es)
    orc = [_engine(oracle_fns, sc) for sc in scs]
    assert len({wd.frame.origin for wd in wds}) >= 30 and len({wd.frame.resolution for wd in wds}) >= 5
    for cycle in range(4):
        resident = cycle >= 2
        outs = (abi.CycleOut * n)()
        bufs = []
        for i in range(n):
            o_i, arrs = es[i]._out()
            outs[i] = o_i
            bufs.append(arrs)
        if resident:
            for e, c in zip(es, cycles):
                e.upload_cycle(c)
            assert product_fns["optimize_batch_resident"](hs, outs, n) == 0, product_fns["last_error"](es[0].h)
        else:
            ins, keep = (abi.CycleIn * n)(), []
            for i, c in enumerate(cycles):
                ins[i], k = c.pack()
                keep.append(k)
            assert product_fns["optimize_batch"](hs, ins, outs, n) == 0, product_fns["last_error"](es[0].h)
        for i in range(n):
            label = f"cycle {cycle} {'resident' if resident else 'batch'} member {i} ({wds[i].frame.name})"
            ro = orc[i].optimize(scs[i].cycle)
            _bars(es[i], orc[i], Engine._result(outs[i], bufs[i]), ro, len(scs[i].critics), label)
            _own_cells(es[i], wds[i].frame, label)
            es[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    assert sum((o.get_cells() == -1).any() for o in orc) >= 15
    for e in es + orc:
        e.close()


def test_group_device_inputs_follow_frame_changes(product_fns, oracle_fns):
    """mppi_optimize_group_device over five cycles in which only the origins move (one cell), then only one member's
    resolution, then only one member's window size changes: bit for bit what mppi_optimize_batch computes from the same
    inputs in host memory, record bytes included, and the oracle's bars.  A member record template that outlived a change
    of its map's geometry would carry the old origin or resolution into the cycle."""
    n = 8
    wds = [mf.world(mf.FRAMES[name], seed=200 + i) for i, name in enumerate(FRAMES)]
    scs = [scenarios.Scenario(f"m{i}", scenarios._omni_cfg(512, 56), scenarios.omni_default_critics(True), _circle_robot(),
                              wd.cycle(), 2000 + i) for i, wd in enumerate(wds)]
    host = [_engine(product_fns, sc, device_map=True) for sc in scs]
    dev = [_engine(product_fns, sc, device_map=True) for sc in scs]
    orc = [_engine(oracle_fns, sc) for sc in scs]
    hh, _ = _bind(product_fns, host), _bind(product_fns, dev)
    changed = set()
    for cycle in range(5):
        if cycle == 1:     # every origin one cell on, nothing else
            wds = [dataclasses.replace(wd, frame=wd.frame.moved(mf.grid_point(wd.frame, 1, -1))) for wd in wds]
        elif cycle == 2:   # one member's resolution
            wds[2] = dataclasses.replace(wds[2], frame=wds[2].frame._replace(resolution=0.04))
        elif cycle == 3:   # one member's window size
            wds[5] = dataclasses.replace(wds[5], frame=wds[5].frame._replace(size_x=wds[5].frame.size_x + 7))
        host_cycles = [wd.cycle() for wd in wds]
        cycles = [_on_device(c) for c in host_cycles]
        changed.add(tuple(wd.frame for wd in wds))
        rh = _host_batch(product_fns, host, hh, cycles)
        rd = optimize_group_device(dev, *_inputs(cycles))
        for i in range(n):
            label = f"cycle {cycle} member {i} ({wds[i].frame.name})"
            _same(host[i], dev[i], rh[i], rd[i], label)
            ro = orc[i].optimize(host_cycles[i])
            _bars(dev[i], orc[i], rd[i], ro, len(scs[i].critics), label)
            _own_cells(dev[i], wds[i].frame, label)
            for e in (host[i], dev[i]):
                e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    assert len(changed) == 4
    for e in host + dev + orc:
        e.close()

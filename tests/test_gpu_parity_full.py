"""Oracle-vs-CUDA parity at the FULL sizes of BASELINE.json configs[2], [3], [4] and for the reference branches the
reduced cases never reach (round-1 verdict, items 1a-1d).

Bars: cell indices and trajectories bit-exact; per-critic costs, total costs and the control sequence within 1e-4
relative.  Absolute floors: 1e-6 on the controls; on costs the floor is COST_ATOL, justified in
profiles/r02b_parity_margins.txt (scripts/parity_margins.py) (the only sums with cancellation are the gamma terms, whose operands are O(1)).
The oracle needs ~25 ms (16384 x 56), ~1 s (262144 x 100) and ~3 ms (2000 x 56) per cycle on one host core.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, abi, scenarios

pytestmark = pytest.mark.gpu

RTOL, ATOL, COST_ATOL = 1e-4, 1e-6, 2e-6


def _engine(fns, sc, noise=None, outputs=True, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise is not None:
        e.set_noise(*noise)
    if outputs:
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    return e


def _compare(g, o, sc, rg, ro, label, bitwise=True):
    if bitwise:
        cg, co = g.get_cells(), o.get_cells()
        assert np.array_equal(cg, co), f"{label}: {np.count_nonzero(cg != co)} cell indices differ"
        for name, a, b in zip("x y yaw".split(), g.get_trajectories(), o.get_trajectories()):
            assert np.array_equal(a, b), f"{label}: trajectory {name} differs in {np.count_nonzero(a != b)} places"
        for q in range(len(sc.critics)):
            np.testing.assert_allclose(g.get_critic_costs(q), o.get_critic_costs(q), rtol=RTOL, atol=COST_ATOL,
                                       err_msg=f"{label}: critic {q} {sc.critics[q][0]}")
    np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=COST_ATOL, err_msg=f"{label}: total costs")
    for name, a, b in (("vx", rg.vx, ro.vx), ("vy", rg.vy, ro.vy), ("wz", rg.wz, ro.wz)):
        np.testing.assert_allclose(a, b, rtol=RTOL, atol=ATOL, err_msg=f"{label}: control {name}")
    assert bool(rg.fail_flag) == bool(ro.fail_flag), label
    assert rg.furthest_reached_path_point == ro.furthest_reached_path_point, label


# ------------------------------------------------------------------------------------------------
# 1a. full sizes
# ------------------------------------------------------------------------------------------------
def test_config3_full_size_against_the_oracle(product_fns, oracle_fns):
    """BASELINE configs[2] as benchmarked: 16384 x 56, 400 x 400 map, ObstaclesCritic in footprint mode (stream layout)."""
    sc = scenarios.config3()
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    for cycle in range(3):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"config3 cycle {cycle}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    c = o.get_critic_costs(0)
    assert (c >= 1e4).any() and (c < 1e4).any() and (c > 0).sum() > 1000   # colliding, free and repelled trajectories
    g.close(); o.close()


def test_config3_dense_footprint_branch_full_size(product_fns, oracle_fns):
    """configs[2] with the robot boxed in (rectangular footprint inside a ring of discs, scenarios.config3(dense=True)):
    the footprint branch of ObstaclesCritic (obstacles_critic.cpp:214-220) is taken by more than a tenth of the visited
    poses in every cycle, more than half of the trajectories collide and break early - the geometry bench.py times as
    obstacles_dense_16384x56."""
    sc = scenarios.config3(dense=True)
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    counters = (C.c_uint64 * 4)()
    for cycle in range(4):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"config3 dense cycle {cycle}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        oracle_fns["get_counters"](o.h, counters)
        assert counters[3] > 0.08 * counters[2] > 0, (cycle, list(counters))
    c = o.get_critic_costs(0)
    assert (c >= 1e4).sum() > 1000 and (c < 1e4).sum() > 1000
    g.close(); o.close()


def _controls_dev(ra, rb):
    """largest relative deviation of the control sequences (floor 1e-6 absolute, the floor of the parity bar)"""
    worst = 0.0
    for name in ("vx", "vy", "wz"):
        a, b = np.asarray(getattr(ra, name), np.float64), np.asarray(getattr(rb, name), np.float64)
        worst = max(worst, float(np.max(np.maximum(np.abs(a - b) - ATOL, 0.0) / np.maximum(np.abs(b), 1e-12))))
    return worst


def test_config4_full_size_against_the_oracle(product_fns, oracle_fns):
    """BASELINE configs[3] on ONE GPU: 262144 x 100, default critic set, 400 x 400 map, N = 120.  The noise is drawn by the
    Philox kernel and handed to the oracle (mppi_get_noise -> oracle set_noise), so both sides see identical bits.

    Cells, trajectories, per-critic costs and total costs: against the oracle as everywhere else.  Control sequence: the
    reference types the softmax normaliser and the weighted sums as float and leaves their order to xtensor/xsimd under
    -ffast-math (optimizer.cpp:384-391).  At 262144 trajectories a float accumulator in index order drops the softmax tail
    (terms below half an ulp of the running sum): the literal index-order oracle itself sits ~3e-4 from the order-free value,
    i.e. two legal evaluation orders of the reference differ by more than the 1e-4 bar.  The bar is therefore applied against
    the oracle with order-free (double) accumulators; the index-order float oracle runs beside it and the test requires the
    device result to be CLOSER to the order-free value than the index-order one is, and within 1e-3 of the latter."""
    sc = scenarios.config4()
    g = _engine(product_fns, sc, None, seed=3)
    g.generate_noise(0)
    noise = g.get_noise()
    o = _engine(oracle_fns, sc, noise)
    oracle_fns["set_wide_reductions"](o.h, 1)
    lit = _engine(oracle_fns, sc, noise, outputs=False)          # literal restatement: float accumulators, index order
    report = []
    for cycle in range(2):
        rg, ro, rl = g.optimize(sc.cycle), o.optimize(sc.cycle), lit.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"config4 cycle {cycle}")
        d_dev, d_lit, d_dev_lit = _controls_dev(rg, ro), _controls_dev(rl, ro), _controls_dev(rg, rl)
        report.append((cycle, d_dev, d_lit, d_dev_lit))
        assert d_dev < d_lit or d_lit < 1e-5, (d_dev, d_lit)
        assert d_dev_lit < 1e-3, d_dev_lit
        for e in (g, lit):
            e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    print("config4 control deviations (cycle, device vs order-free, index-order float vs order-free, device vs index-order):", report)
    # what bench.py times: nothing materialised (exact instance), same controls
    g.set_outputs()
    g.set_control_sequence(*(np.zeros(100, np.float32),) * 3)
    o.set_control_sequence(*(np.zeros(100, np.float32),) * 3)
    rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
    _compare(g, o, sc, rg, ro, "config4, no outputs", bitwise=False)
    g.close(); o.close(); lit.close()


@pytest.mark.parametrize("mode", ["stream"])
def test_config5_every_member_of_a_bound_group_against_the_oracle(product_fns, oracle_fns, mode):
    """BASELINE configs[4]: robots of 2000 x 56 with their own map / path / heading, served as ONE bound group
    (mppi_batch_bind): every member's controls, costs, flag and furthest point against its own oracle, 4 cycles."""
    ids = [0, 1, 37, 64, 100, 128, 129, 191, 200, 255]
    scs = [scenarios.config5_robot(r) for r in ids]
    n, T = len(scs), scs[0].cfg["time_steps"]
    group = [_engine(product_fns, sc, sc.noise(), outputs=False) for sc in scs]
    orcs = [_engine(oracle_fns, sc, sc.noise(), outputs=False) for sc in scs]
    hs = (abi.H * n)(*[e.h for e in group])
    assert product_fns["batch_bind"](hs, n) == 0
    ins, outs = (abi.CycleIn * n)(), (abi.CycleOut * n)()
    keep, bufs = [], []
    for i, sc in enumerate(scs):
        cin, k = sc.cycle.pack()
        ins[i] = cin
        arrs = [np.empty(T, np.float32) for _ in range(3)]
        outs[i].control_vx, outs[i].control_vy, outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
        keep.append(k); bufs.append(arrs)
    launches0 = sum(e.get_profile()["kernel_launches"] for e in group)
    for cycle in range(4):
        assert product_fns["optimize_batch"](hs, ins, outs, n) == 0
        for i, (sc, o) in enumerate(zip(scs, orcs)):
            ro = o.optimize(sc.cycle)
            for a, name in zip(bufs[i], ("vx", "vy", "wz")):
                np.testing.assert_allclose(a, getattr(ro, name), rtol=RTOL, atol=ATOL, err_msg=f"cycle {cycle} robot {ids[i]} {name}")
            assert bool(outs[i].fail_flag) == bool(ro.fail_flag)
            want = abi.UINT32_MAX if ro.furthest_reached_path_point is None else ro.furthest_reached_path_point
            assert outs[i].furthest_reached_path_point == want
            np.testing.assert_allclose(group[i].get_costs(), o.get_costs(), rtol=RTOL, atol=COST_ATOL,
                                       err_msg=f"cycle {cycle} robot {ids[i]} costs")
            group[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    n_launches = sum(e.get_profile()["kernel_launches"] for e in group) - launches0
    assert n_launches <= 4 * 4, n_launches   # the group really ran as a group: <= 4 launches per cycle for all robots
    # one member on its own with everything materialised: bit-exact cells and trajectories
    g, o, sc = group[3], orcs[3], scs[3]
    for e in (g, o):
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
    _compare(g, o, sc, rg, ro, f"robot {ids[3]} alone")
    for e in group + orcs:
        e.close()


# ------------------------------------------------------------------------------------------------
# 1b. getOptimizedTrajectory (optimizer.cpp:345-360 -> :275-311)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["Omni", "DiffDrive"])
def test_optimized_trajectory_against_the_oracle(product_fns, oracle_fns, model):
    sc = scenarios.config1(batch=512)
    sc.cfg["motion_model"] = model
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise, outputs=False), _engine(oracle_fns, sc, noise, outputs=False)
    pose = (sc.cycle.pose[0], sc.cycle.pose[1], 0.7)
    cyc = dataclasses.replace(sc.cycle, pose=pose)
    for cycle in range(6):
        rg, ro = g.optimize(cyc), o.optimize(cyc)
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        tg, to = g.get_optimized_trajectory(pose), o.get_optimized_trajectory(pose)
        assert tg.shape == (sc.cfg["time_steps"], 3)
        assert np.array_equal(tg, to), f"cycle {cycle}: {np.count_nonzero(tg != to)} elements differ"
    assert np.abs(to[-1, :2] - np.asarray(pose[:2])).max() > 0.05   # the sequence moves the robot
    g.close(); o.close()


# ------------------------------------------------------------------------------------------------
# 1c. reference branches that no other test reaches
# ------------------------------------------------------------------------------------------------
def _near_obstacle_map(unknown=False):
    """config1's discs keep clear of the robot; these two sit 0.4 - 0.6 m from it so that sampled trajectories run through
    inflated, inscribed and lethal cells from the first cycle on (robot at cell (50, 50), path along +x)"""
    cm = scenarios.inflated_disc_costmap(100, 100, 0.05, [(57.0, 55.5, 2.5), (62.0, 44.0, 2.0)])
    if unknown:
        cm[49:52, 75:78] = 255          # ON the path: path points 25..27 sit in unknown space (utils.hpp:386-388)
        cm[46:49, 53:58] = 255          # beside the path, 0.15 - 0.4 m ahead: trajectories wander through it
        cm[53:55, 51:54] = 255          # and a patch on the other side, inside the first disc's inflation
    return cm


def _with_critic(sc, name, **kw):
    out = []
    for cname, params in sc.critics:
        out.append((cname, dict(params, **kw)) if cname == name else (cname, params))
    sc.critics = out
    return sc


@pytest.mark.parametrize("layout", ["tile", "stream"])
def test_path_angle_reversing_branch(product_fns, oracle_fns, monkeypatch, layout):
    """forward_preference = false with vx_min < 0 (path_angle_critic.cpp:36-40,92-97, utils.hpp:417-434): the bearing is
    corrected by +-pi when that is the shorter way.  Robot facing AWAY from the path: with forward preference the gate is
    open and the critic fires, with the reversing branch the corrected bearing is small; poses sideways on fire either way."""
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1" if layout == "stream" else "1000000000")
    fired = {}
    for yaw in (1.9, 2.9):
        sc = _with_critic(scenarios.config1(batch=512), "PathAngleCritic", forward_preference=0)
        sc.cycle.pose = (sc.cycle.pose[0], sc.cycle.pose[1], yaw)
        sc.cycle.speed = (-0.2, 0.05, 0.1)
        noise = sc.noise()
        g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
        for cycle in range(3):
            rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
            _compare(g, o, sc, rg, ro, f"reversing yaw {yaw} cycle {cycle}")
            g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        idx = [c[0] for c in sc.critics].index("PathAngleCritic")
        fired[yaw] = float(o.get_critic_costs(idx).max())
        g.close(); o.close()
    assert fired[1.9] > 0.0          # 1.9 rad off forwards, pi - 1.9 = 1.24 rad off backwards: above max_angle (1.0) both ways
    assert fired[2.9] == 0.0         # backing up along the path: the corrected bearing (0.24 rad) closes the gate
    # the same pose WITH forward preference fires: the two branches really differ
    sc = scenarios.config1(batch=512)
    sc.cycle.pose = (sc.cycle.pose[0], sc.cycle.pose[1], 2.9)
    o = _engine(oracle_fns, sc, sc.noise())
    o.optimize(sc.cycle)
    assert o.get_critic_costs([c[0] for c in sc.critics].index("PathAngleCritic")).max() > 0.0
    o.close()


@pytest.mark.parametrize("layout", ["tile", "stream"])
def test_path_align_use_path_orientations(product_fns, oracle_fns, monkeypatch, layout):
    """use_path_orientations = true (path_align_critic.cpp:119-123; legacy :108-113): the yaw distance to the path point
    joins the positional one.  A curved path so that the path yaws differ from point to point."""
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1" if layout == "stream" else "1000000000")
    sc = _with_critic(scenarios.config1(batch=512), "PathAlignCritic", use_path_orientations=1, offset_from_furthest=6)
    sc.critics.append(("PathAlignLegacyCritic", dict(use_path_orientations=1, offset_from_furthest=6)))
    s = np.arange(40) * 0.05
    yaw = 0.6 * s
    px = (sc.cycle.pose[0] + np.cumsum(np.cos(yaw)) * 0.05 - 0.05).astype(np.float32)
    py = (sc.cycle.pose[1] + np.cumsum(np.sin(yaw)) * 0.05).astype(np.float32)
    sc.cycle = dataclasses.replace(sc.cycle, path_x=px, path_y=py, path_yaw=yaw.astype(np.float32),
                                   goal=(float(px[-1]), float(py[-1])), costmap=np.zeros_like(sc.cycle.costmap))
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    plain = _engine(oracle_fns, _with_critic(dataclasses.replace(sc, critics=list(sc.critics)), "PathAlignCritic", use_path_orientations=0), noise)
    for cycle in range(14):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        plain.optimize(sc.cycle)
        if cycle in (0, 1, 8, 13):
            _compare(g, o, sc, rg, ro, f"use_path_orientations cycle {cycle}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        plain.set_control_sequence(ro.vx, ro.vy, ro.wz)
    idx = [c[0] for c in sc.critics].index("PathAlignCritic")
    a, b = o.get_critic_costs(idx), plain.get_critic_costs(idx)
    assert a.max() > 0.0 and (a > b + 1e-3).any()     # the critic ran and the yaw term changed its value
    assert o.get_critic_costs(len(sc.critics) - 1).max() > 0.0
    for e in (g, o, plain):
        e.close()


@pytest.mark.parametrize("layout", ["tile", "stream"])
@pytest.mark.parametrize("footprint", [True, False])
def test_track_unknown_with_no_information_cells(product_fns, oracle_fns, monkeypatch, layout, footprint):
    """track_unknown = true (cost_critic.cpp:195, obstacles_critic.cpp:197, utils.hpp:386-388): NO_INFORMATION (255) cells
    under the trajectories and ON the path are costs, not collisions, and do not invalidate path points; with
    track_unknown = false the same map makes trajectories collide and path points invalid."""
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1" if layout == "stream" else "1000000000")
    got = {}
    for track in (1, 0):
        sc = scenarios.config1(batch=512, cost_consider_footprint=footprint)
        sc.critics.append(("ObstaclesCritic", dict(consider_footprint=int(footprint), cost_scaling_factor=3.0)))
        cm = _near_obstacle_map(unknown=True)
        sc.cycle = dataclasses.replace(sc.cycle, costmap=cm, speed=(0.3, 0.0, 0.0))
        sc.robot.track_unknown = track
        noise = sc.noise()
        g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
        for cycle in range(10):
            rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
            if cycle in (0, 1, 9):
                _compare(g, o, sc, rg, ro, f"track_unknown={track} cycle {cycle}")
            if cycle == 0:   # same inputs for both settings: comparable counts
                got[track] = (o.get_critic_costs(1).copy(), o.get_critic_costs(len(sc.critics) - 1).copy())
            g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        cells = o.get_cells()
        assert (cm.reshape(-1)[cells[cells >= 0]] == 255).any()       # trajectories did cross unknown cells
        g.close(); o.close()
    # a collided trajectory costs 3.81 / 254 * 1e6 / 56 = 267.86 (CostCritic) and 20 * 1e4 = 2e5 (ObstaclesCritic)
    assert (got[0][0] > 200.0).sum() > (got[1][0] > 200.0).sum() > 0  # unknown cells collide only when not tracked
    assert (got[0][1] >= 1e5).sum() > (got[1][1] >= 1e5).sum() > 0


@pytest.mark.parametrize("layout", ["tile", "stream"])
def test_no_inflation_layer_in_footprint_mode(product_fns, oracle_fns, monkeypatch, layout):
    """inflation_layer_found = false with consider_footprint = true (cost_critic.cpp:63-106, obstacles_critic.cpp:53-97):
    findCircumscribedCost returns -1 -> possibly_inscribed_cost < 1 -> the footprint is checked at EVERY costed pose, and the
    Obstacles critic runs with its default scale / radius (inflation_radius 0, cost_scaling_factor 0 -> no repulsion)."""
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1" if layout == "stream" else "1000000000")
    sc = scenarios.config1(batch=512, footprint="bowtie")
    sc.critics.append(("ObstaclesCritic", dict(consider_footprint=1)))
    sc.robot.inflation_layer_found = 0
    sc.cycle = dataclasses.replace(sc.cycle, costmap=_near_obstacle_map(), speed=(0.3, 0.0, 0.0))
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    for cycle in range(4):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"no inflation layer cycle {cycle}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    c = o.get_critic_costs(1)
    assert (c > 200.0).any() and ((c > 0.0) & (c < 200.0)).any()    # collided (267.86) and merely costed trajectories
    g.close(); o.close()


# ------------------------------------------------------------------------------------------------
# 1e. the stream layout's furthest-point scan (skips along the path) and lean per-trajectory total
# ------------------------------------------------------------------------------------------------
def _winding_paths(x0, y0):
    """paths on which the distance to a pose is NOT unimodal along the path, with ties, repeated points, uneven spacing"""
    out = {}
    s = np.linspace(0.0, 1.0, 90)
    # a loop that leaves the robot, comes back past it and leaves again: several local minima
    out["loop"] = (x0 + 1.2 * np.sin(2 * np.pi * s) + 0.8 * s, y0 + 0.9 * (1 - np.cos(2 * np.pi * s)) * np.sign(0.5 - s + 1e-9))
    # out and back along the SAME line: every distance appears twice (ties -> the first index must win)
    leg = np.arange(30) * 0.05
    out["out_and_back"] = (x0 + np.concatenate([leg, leg[::-1]]), np.full(60, y0))
    # uneven spacing: repeated points (zero-length segments), then a 0.6 m jump, then dense points
    xs = np.concatenate([np.zeros(4), np.arange(1, 12) * 0.03, 0.33 + 0.6 + np.arange(25) * 0.01, 1.2 + np.arange(10) * 0.2])
    out["uneven"] = (x0 + xs, y0 + 0.1 * np.sin(5 * xs))
    # a spiral around the robot
    th = np.linspace(0.0, 5 * np.pi, 120)
    out["spiral"] = (x0 + (0.1 + 0.09 * th) * np.cos(th), y0 + (0.1 + 0.09 * th) * np.sin(th))
    return {k: (np.asarray(a, np.float32), np.asarray(b, np.float32)) for k, (a, b) in out.items()}


@pytest.mark.parametrize("shape", ["loop", "out_and_back", "uneven", "spiral"])
def test_stream_layout_on_winding_paths(product_fns, oracle_fns, monkeypatch, shape):
    """utils::findPathFurthestReachedPoint (utils.hpp:292-319) is a first-minimum scan over ALL path points; the stream
    kernel skips points that provably cannot win.  Paths with several local minima, exact ties, repeated points and uneven
    spacing: furthest point, per-critic costs, total costs and controls against the oracle; then the same without
    materialised outputs (the lean per-trajectory total of the path-cost kernel)."""
    monkeypatch.setenv("MPPI_STREAM_MIN_BATCH", "1")
    sc = scenarios.config1(batch=2048)
    px, py = _winding_paths(sc.cycle.pose[0], sc.cycle.pose[1])[shape]
    pyaw = np.arctan2(np.gradient(py.astype(np.float64)), np.gradient(px.astype(np.float64)) + 1e-12).astype(np.float32)
    sc.cycle = dataclasses.replace(sc.cycle, path_x=px, path_y=py, path_yaw=pyaw, goal=(float(px[-1]) + 3.0, float(py[-1])),
                                   costmap=np.zeros_like(sc.cycle.costmap), speed=(0.25, 0.05, 0.1))
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    seen = set()
    for cycle in range(5):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"{shape} cycle {cycle}")
        seen.add(ro.furthest_reached_path_point)
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    assert None not in seen
    g.set_outputs(); o.set_outputs()
    for cycle in range(3):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _compare(g, o, sc, rg, ro, f"{shape} lean cycle {cycle}", bitwise=False)
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    g.close(); o.close()


def test_stream_layout_is_deterministic_over_repeated_cycles(product_fns):
    """The stream layout's last kernel merges its own partial records (the block that finishes a row group last sums that
    group's columns): a race there would show as a result that changes from run to run.  The same cycle 40 times from the
    same control sequence: identical bits every time."""
    sc = scenarios.config4(batch=65536)
    g = _engine(product_fns, sc, None, outputs=False, seed=3)
    g.generate_noise(0)
    zero = np.zeros(sc.cfg["time_steps"], np.float32)
    first = None
    for cycle in range(40):
        g.set_control_sequence(zero, zero, zero)
        r = g.optimize(sc.cycle)
        got = np.concatenate([r.vx, r.vy, r.wz])
        if first is None:
            first = got.copy()
            assert np.abs(first).max() > 1e-3
        assert np.array_equal(got, first), f"cycle {cycle}: {np.count_nonzero(got != first)} of {got.size} values changed"
    g.close()

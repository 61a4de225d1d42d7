"""The reference the map-frame GPU tests (test_gpu_map_frames.py) compare against, and their helpers, checked on the CPU:
the oracle's worldToMap and its rollout cells equal cells_fp64 on offset, negative, non-square, non-0.05 m frames; the
rolling window keeps its origin on the grid; every frame's path leaves the window; edge_poses reaches the poses whose
fp32 cell is not their fp64 cell."""
import ctypes as C

import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, abi, scenarios
from mpcholonavigation_b200.api import circle_footprint, make_robot
from tests import map_frames as mf

FRAMES = list(mf.FRAMES)


def test_frames_are_what_they_claim():
    for f in mf.FRAMES.values():
        assert any(float(np.float32(o)) != o for o in f.origin), f.name   # fl32(origin) is not the origin
    assert mf.FRAMES["odom"].size_x * mf.FRAMES["odom"].size_y % 16 != 0
    assert mf.FRAMES["big_window"].size_x * mf.FRAMES["big_window"].size_y > 96 * 1024
    assert float(np.float32(1.0 / 0.03)) != 1.0 / 0.03
    assert all(e >= 0.5 for e in mf.cell_eps(mf.FRAMES["filter_off"]))
    assert all(e < 0.5 for f in mf.FRAMES.values() if f.name != "filter_off" for e in mf.cell_eps(f))


@pytest.mark.parametrize("frame", FRAMES)
def test_oracle_world_to_map_is_cells_fp64(oracle_fns, frame):
    """Costmap2D::worldToMap of the oracle, pose by pose, on every edge pose of the frame"""
    f = mf.FRAMES[frame]
    p = mf.edge_poses(f)
    cm = abi.Costmap()
    cells = np.zeros((f.size_y, f.size_x), np.uint8)
    cm.cells = cells.ctypes.data_as(abi.u8p)
    cm.size_x, cm.size_y, cm.resolution = f.size_x, f.size_y, f.resolution
    cm.origin_x, cm.origin_y = f.origin
    w2m = oracle_fns["world_to_map"]
    got = np.array([w2m(C.byref(cm), float(x), float(y)) for x, y in zip(p.x.tolist(), p.y.tolist())], np.int32)
    want = mf.cells_fp64(p.x, p.y, f)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} poses, first ({p.x[bad[0]]!r}, {p.y[bad[0]]!r}): {got[bad[0]]} vs {want[bad[0]]}"
    assert (want == -1).any() and (want >= 0).any()


@pytest.mark.parametrize("frame", FRAMES)
def test_oracle_rollout_cells_are_cells_fp64(oracle_fns, frame):
    """oracle optimize() on the frame's world: the cell of every rollout pose is cells_fp64 of that pose"""
    wd = mf.world(mf.FRAMES[frame], seed=3)
    cfg = scenarios._omni_cfg(128, 56)
    e = Engine(oracle_fns, **cfg)
    e.set_robot(make_robot(circle_footprint(0.25), inscribed_radius=0.25, circumscribed_radius=0.25,
                           inflation_layer_found=True, inflation_cost_scaling_factor=3.0))
    e.set_critics(scenarios.omni_default_critics(True))
    e.set_outputs(trajectories=True, cells=True)
    rng = np.random.default_rng(0)
    e.set_noise(*(rng.standard_normal((128, 56)).astype(np.float32) * s for s in (0.6, 0.6, 0.4)))
    e.optimize(wd.cycle())
    x, y, _ = e.get_trajectories()
    assert np.array_equal(e.get_cells(), mf.cells_fp64(x, y, wd.frame))
    e.close()


@pytest.mark.parametrize("frame", FRAMES)
def test_edge_poses_reach_their_targets(frame):
    f = mf.FRAMES[frame]
    p = mf.edge_poses(f)
    c64 = mf.cells_fp64(p.x, p.y, f)
    cand, sure = mf.filter_fp32(p.x, p.y, f)
    # the mirror of the device's filter never claims a cell it would get wrong
    assert not (sure & (cand != c64)).any()
    if frame == "filter_off":
        assert not sure.any()
    else:
        assert sure.mean() > 0.75
    if frame != "res_01":   # at 0.1 m, fl32(origin) moves every fp32 edge onto a pose value, never across one
        assert (cand != c64).any(), "no pose whose fp32 cell differs from its fp64 cell"
    for key, (below, above) in mf.edge_sides(p, f).items():
        assert below > 0 and above > 0, key
    kinds = set(p.kind.tolist())
    assert kinds == set(range(len(mf.KINDS)))
    off = p.kind == mf.KINDS.index("off_map")
    assert (c64[off] == -1).all()


@pytest.mark.parametrize("frame", FRAMES)
def test_paths_leave_the_window(frame):
    wd = mf.world(mf.FRAMES[frame], seed=3)
    c = mf.cells_fp64(wd.path_x, wd.path_y, wd.frame)
    assert c[0] >= 0 and (c == -1).any()
    assert mf.cells_fp64(np.float32([wd.pose[0]]), np.float32([wd.pose[1]]), wd.frame)[0] >= 0


@pytest.mark.parametrize("frame", ["odom", "campus", "res_003"])
def test_rolling_keeps_the_origin_on_the_grid(frame):
    f0 = mf.FRAMES[frame]
    wd = mf.world(f0, seed=1)
    x, y, yaw = wd.pose
    moved = 0
    for k in range(40):
        x, y = x + 0.137 * np.cos(yaw), y + 0.137 * np.sin(yaw)
        nxt = mf.rolling(wd, (x, y, yaw))
        moved += nxt.frame.origin != wd.frame.origin
        wd = nxt
        for a in (0, 1):
            q = (wd.frame.origin[a] - f0.origin[a]) / f0.resolution
            assert abs(q - round(q)) < 1e-6, (k, a, q)
        cx, cy = wd.frame.centre
        assert abs(cx - x) <= f0.resolution and abs(cy - y) <= f0.resolution
        assert wd.costmap().shape == (f0.size_y, f0.size_x)
    assert moved >= 30

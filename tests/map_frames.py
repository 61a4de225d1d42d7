"""Costmaps away from the world origin: offset and negative origins, non-square windows, resolutions other than 0.05 m,
and the rolling window of Nav2's local costmap.  TEST INFRASTRUCTURE: nothing under mpcholonavigation_b200/ imports this.

The kernels map a rollout pose to a cell with an fp32 filter (mppi_device.cuh world_to_cell_fast): the fp32 candidate
is taken only when it is farther from a cell edge than an error bound that build_params derives from the origin, the
resolution and the map size; otherwise the reference's fp64 worldToMap decides.  With the origin at (0, 0), 0.05 m cells
and square maps, the origin term of that bound is zero, fl32(1/res) is exact and x / y are interchangeable, so the
frames below are chosen to make each of those parts matter.

cells_fp64 is the independent reference for every cell check (Costmap2D::worldToMap restated in numpy); filter_fp32
mirrors the device's filter and is used only to assert that a test reached the poses it is about.
"""
import dataclasses
from typing import NamedTuple, Tuple

import numpy as np

from mpcholonavigation_b200 import scenarios
from mpcholonavigation_b200.api import Cycle

F32 = np.float32


class Frame(NamedTuple):
    name: str
    origin: Tuple[float, float]
    resolution: float
    size_x: int
    size_y: int

    @property
    def extent(self):
        return self.size_x * self.resolution, self.size_y * self.resolution

    @property
    def centre(self):
        return (self.origin[0] + self.size_x * self.resolution / 2.0, self.origin[1] + self.size_y * self.resolution / 2.0)

    def moved(self, origin):
        return self._replace(origin=(float(origin[0]), float(origin[1])))


# every origin is a double that fp32 does not hold exactly
FRAMES = {f.name: f for f in (
    Frame("odom", (12.35, -48.65), 0.05, 121, 87),                       # odd, non-square, zero-copy upload
    Frame("far_negative", (-1234.567, -987.65), 0.05, 160, 100),
    Frame("res_003", (3.21, 7.77), 0.03, 200, 150),                      # fl32(1 / 0.03) is not 1 / 0.03
    Frame("res_007_tall", (-5.5, 20.05), 0.07, 64, 180),
    Frame("res_01", (250.05, -300.15), 0.1, 100, 60),
    Frame("campus", (8123.4, -4210.7), 0.05, 120, 120),                  # the origin term dominates the bound
    Frame("big_window", (-20.025, 40.075), 0.05, 401, 263),              # 105 KB: above the zero-copy bound
    Frame("filter_off", (1.0e5 + 0.013, -1.0e5 - 0.007), 0.01, 90, 70),  # 0.5 - cell_eps <= 0: every pose takes fp64
)}


# ------------------------------------------------------------------------------------------------
# cell arithmetic
# ------------------------------------------------------------------------------------------------
def axis_cells_fp64(v, o, res, size):
    """worldToMap on one axis, in fp64: the cell index, -1 below the origin, `size` at or beyond the far edge."""
    w = np.asarray(v, np.float32).astype(np.float64)
    q = (w - float(o)) / float(res)
    idx = np.full(w.shape, -1, np.int64)
    on = ~(w < float(o))
    idx[on & ~(q < float(size))] = size
    inside = on & (q < float(size))
    idx[inside] = np.trunc(q[inside]).astype(np.int64)
    return idx


def cells_fp64(x, y, frame):
    """Costmap2D::worldToMap for fp32 poses widened to double: `wx < ox` test, fp64 quotient, truncation; the flat index
    my * size_x + mx, or -1 off the map."""
    ox, oy = frame.origin
    mx = axis_cells_fp64(x, ox, frame.resolution, frame.size_x)
    my = axis_cells_fp64(y, oy, frame.resolution, frame.size_y)
    on = (mx >= 0) & (mx < frame.size_x) & (my >= 0) & (my < frame.size_y)
    return np.where(on, my * frame.size_x + mx, -1).astype(np.int32)


def cell_eps(frame):
    """build_params' error bounds of the fp32 filter, in cells, as the fp32 values the kernels read."""
    u = 2.0 ** -24
    ox, oy = frame.origin
    res = frame.resolution
    ex = F32(((frame.size_x + 2.0) * 3.5 + abs(ox) / res * 1.1) * u + 1.0e-6)
    ey = F32(((frame.size_y + 2.0) * 3.5 + abs(oy) / res * 1.1) * u + 1.0e-6)
    return ex, ey


def _add_round_down(q, c):
    """fl32 of q + c rounded toward -inf (__fadd_rd): the exact sum in fp64, then the fp32 at or below it."""
    s = q.astype(np.float64) + float(c)
    f = s.astype(np.float32)
    return np.where(f.astype(np.float64) > s, np.nextafter(f, F32(-np.inf)), f)


def _floor_magic(q):
    t = _add_round_down(q, F32(12582912.0))
    i = t.view(np.int32).astype(np.int64) - 0x4B400000
    frac = (q - (t - F32(12582912.0))).astype(np.float32)
    return i, frac


def filter_fp32(x, y, frame):
    """The device's fp32 filter (world_to_cell_try) in IEEE fp32: (candidate flat cell or -1, sure).  For coverage
    assertions only: where `sure` is False the device takes the fp64 path, so the candidate is not its answer."""
    with np.errstate(over="ignore", invalid="ignore"):
        xf, yf = np.asarray(x, F32), np.asarray(y, F32)
        oxf, oyf = F32(frame.origin[0]), F32(frame.origin[1])
        invf = F32(1.0 / frame.resolution)
        qx = ((xf - oxf).astype(F32) * invf).astype(F32)
        qy = ((yf - oyf).astype(F32) * invf).astype(F32)
        mx, fx = _floor_magic(qx)
        my, fy = _floor_magic(qy)
        ex, ey = cell_eps(frame)
        hx, hy = (F32(0.5) - ex).astype(F32), (F32(0.5) - ey).astype(F32)
        sure = (np.abs((fx - F32(0.5)).astype(F32)) < hx) & (np.abs((fy - F32(0.5)).astype(F32)) < hy)
    on = (mx >= 0) & (mx < frame.size_x) & (my >= 0) & (my < frame.size_y)
    return np.where(on, my * frame.size_x + mx, -1).astype(np.int32), sure


def grid_point(frame, kx, ky):
    """the world point of cell corner (kx, ky), in double, as the costmap defines it"""
    return frame.origin[0] + kx * frame.resolution, frame.origin[1] + ky * frame.resolution


# ------------------------------------------------------------------------------------------------
# poses around cell edges
# ------------------------------------------------------------------------------------------------
class EdgePoses(NamedTuple):
    x: np.ndarray       # fp32
    y: np.ndarray       # fp32
    kind: np.ndarray    # KINDS index
    axis: np.ndarray    # 0: the x edge `edge` is tested, 1: the y edge, 2: both (a corner), -1: none
    edge: np.ndarray    # the edge index on the tested axis (0 .. size), -1 if none


KINDS = ("interior", "origin", "far", "corner", "random", "off_map")


def _ulps_around(v, n):
    """the 2n+1 fp32 values from n ulps below fl32(v) to n ulps above"""
    f = np.float32(v)
    out = [f]
    lo = hi = f
    for _ in range(n):
        lo, hi = np.nextafter(lo, F32(-np.inf)), np.nextafter(hi, F32(np.inf))
        out += [lo, hi]
    return np.sort(np.array(out, F32))


def _interior(frame, rng, n, axis_size, axis):
    res = frame.resolution
    o = frame.origin[axis]
    return (o + rng.uniform(0.02, axis_size - 0.02, n) * res).astype(F32)


def edge_poses(frame, n_ulps=40, total=64512, seed=0, n_interior_edges=None):
    """fp32 poses at -n_ulps .. +n_ulps around: the interior cell edges of both axes (all of them, or n_interior_edges
    drawn at random), the origin edges, the far edges
    (size * res), a few cell corners; then random interior points and far off-map points (|q| from 10 to 2^25 cells, on
    both sides of both axes) up to `total` poses."""
    rng = np.random.default_rng(seed)
    sizes = (frame.size_x, frame.size_y)
    xs, ys, kinds, axes, edges = [], [], [], [], []

    def add(x, y, kind, axis, edge):
        xs.append(np.asarray(x, F32)), ys.append(np.asarray(y, F32))
        n = len(xs[-1])
        kinds.append(np.full(n, KINDS.index(kind))), axes.append(np.full(n, axis)), edges.append(np.full(n, edge))

    for axis in (0, 1):
        size = sizes[axis]
        inner = np.arange(1, size) if n_interior_edges is None else rng.choice(np.arange(1, size), n_interior_edges, replace=False)
        for kind, ks in (("interior", inner), ("origin", [0]), ("far", [size])):
            for k in ks:
                v = _ulps_around(frame.origin[axis] + int(k) * frame.resolution, n_ulps)
                other = _interior(frame, rng, len(v), sizes[1 - axis], 1 - axis)
                add(*((v, other) if axis == 0 else (other, v)), kind, axis, int(k))
    # corners: both coordinates within n_ulps of an edge, every 4th ulp offset
    step = 4
    for kx, ky in [(0, 0), (sizes[0], sizes[1]), (0, sizes[1]), (sizes[0], 0),
                   (int(rng.integers(1, sizes[0])), int(rng.integers(1, sizes[1])))]:
        gx, gy = grid_point(frame, kx, ky)
        vx, vy = _ulps_around(gx, n_ulps)[::step], _ulps_around(gy, n_ulps)[::step]
        X, Y = np.meshgrid(vx, vy)
        add(X.ravel(), Y.ravel(), "corner", 2, -1)
    # far off the map: |q| in [10, 2^25] cells, both sides of both axes
    n_off = 2048
    q = np.exp(rng.uniform(np.log(10.0), np.log(2.0 ** 25), n_off))
    side = rng.integers(0, 2, n_off)
    axis = rng.integers(0, 2, n_off)
    for a in (0, 1):
        m = axis == a
        lo = frame.origin[a] - q[m] * frame.resolution
        hi = frame.origin[a] + (sizes[a] + q[m]) * frame.resolution
        v = np.where(side[m] == 0, lo, hi).astype(F32)
        other = _interior(frame, rng, int(m.sum()), sizes[1 - a], 1 - a)
        add(*((v, other) if a == 0 else (other, v)), "off_map", -1, -1)
    n = sum(len(a) for a in xs)
    assert n <= total, n
    rest = total - n
    add(_interior(frame, rng, rest, sizes[0], 0), _interior(frame, rng, rest, sizes[1], 1), "random", -1, -1)
    return EdgePoses(*(np.concatenate(a) for a in (xs, ys, kinds, axes, edges)))


def edge_sides(poses, frame):
    """{(kind, axis, edge): (poses below the edge, poses at or above it)}, counted in fp64, for the edge kinds"""
    mx = axis_cells_fp64(poses.x, frame.origin[0], frame.resolution, frame.size_x)
    my = axis_cells_fp64(poses.y, frame.origin[1], frame.resolution, frame.size_y)
    out = {}
    for kind in ("interior", "origin", "far"):
        for axis, m in ((0, mx), (1, my)):
            sel = (poses.kind == KINDS.index(kind)) & (poses.axis == axis)
            for k in np.unique(poses.edge[sel]):
                s = sel & (poses.edge == k)
                out[(kind, axis, int(k))] = (int((m[s] < k).sum()), int((m[s] >= k).sum()))
    return out


# ------------------------------------------------------------------------------------------------
# a world seen through a frame
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class World:
    frame: Frame
    discs: list           # (x [m], y [m], r [m]) in world coordinates
    path_x: np.ndarray    # fp32 world coordinates; runs past the window edge
    path_y: np.ndarray
    path_yaw: np.ndarray
    pose: tuple           # (x, y, yaw), world coordinates
    goal: tuple
    inscribed_radius: float = 0.25

    def costmap(self):
        """the discs rasterised into the window, centres converted to window cells"""
        f = self.frame
        ox, oy = f.origin
        cells = [((x - ox) / f.resolution, (y - oy) / f.resolution, r / f.resolution) for x, y, r in self.discs]
        return scenarios.inflated_disc_costmap(f.size_x, f.size_y, f.resolution, cells,
                                               inscribed_radius=self.inscribed_radius)

    def cycle(self, speed=(0.0, 0.0, 0.0)):
        return Cycle(pose=self.pose, speed=speed, goal=self.goal, goal_checker_xy_tolerance=0.25, path_x=self.path_x,
                     path_y=self.path_y, path_yaw=self.path_yaw, costmap=self.costmap(), resolution=self.frame.resolution,
                     origin=self.frame.origin)


def world(frame, seed=0, ring=None, inscribed_radius=0.25, n_path=120, edge_margin=None):
    """Discs and a straight path in world coordinates around a robot near the window centre, or `edge_margin` metres
    inside the window's low-x edge (so that the rollouts leave the map).  The path runs 1.2 window diagonals, so its
    far end is off the map whatever the heading.  ring = r [m]: eight more discs r away from the robot (the boxed-in case
    of scenarios.config3(dense=True))."""
    rng = np.random.default_rng(seed)
    w, h = frame.extent
    cx, cy = frame.centre
    pose = (cx + rng.uniform(-0.1, 0.1) * w, cy + rng.uniform(-0.1, 0.1) * h, float(rng.uniform(-np.pi, np.pi)))
    if edge_margin is not None:
        pose = (frame.origin[0] + min(edge_margin, w / 2.0), pose[1], pose[2])
    length = 1.2 * float(np.hypot(w, h))
    px, py, pyaw = scenarios.straight_path(pose[0], pose[1], pose[2], n_path, length / (n_path - 1))
    keep = min(0.6, 0.3 * min(w, h)) if ring is None else 0.9 * ring
    k = int(np.clip(w * h / 2.0, 4, 60))
    discs, guard = [], 0
    while len(discs) < k and guard < 100000:
        guard += 1
        x, y = frame.origin[0] + rng.uniform(0, w), frame.origin[1] + rng.uniform(0, h)
        r = rng.uniform(0.1, 0.2)
        if np.hypot(x - pose[0], y - pose[1]) >= keep + r:
            discs.append((x, y, r))
    if ring is not None:
        for j in range(8):
            a = 2.0 * np.pi * (j + 0.5) / 8
            discs.append((pose[0] + ring * np.cos(a), pose[1] + ring * np.sin(a), 0.1))
    return World(frame, discs, px, py, pyaw, pose, (float(px[-1]), float(py[-1])), inscribed_radius)


def rolling(wd, pose):
    """Costmap2D::updateOrigin for a window centred on `pose`: the origin moves by whole cells (in double, as Nav2 adds
    cell_o * resolution to the old origin), the map is re-rasterised from the same discs."""
    f = wd.frame
    res = f.resolution
    new_ox, new_oy = pose[0] - f.size_x * res / 2.0, pose[1] - f.size_y * res / 2.0
    cell_ox, cell_oy = int((new_ox - f.origin[0]) / res), int((new_oy - f.origin[1]) / res)
    moved = f.moved((f.origin[0] + cell_ox * res, f.origin[1] + cell_oy * res))
    return dataclasses.replace(wd, frame=moved, pose=tuple(pose))


def prune_path(wd, pose):
    """the path from its point closest to `pose` on (the controller is handed the remaining plan)"""
    d = np.hypot(wd.path_x.astype(np.float64) - pose[0], wd.path_y.astype(np.float64) - pose[1])
    i = int(np.argmin(d))
    i = min(i, len(wd.path_x) - 2)
    return dataclasses.replace(wd, path_x=wd.path_x[i:].copy(), path_y=wd.path_y[i:].copy(), path_yaw=wd.path_yaw[i:].copy())

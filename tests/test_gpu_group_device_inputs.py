"""Robot groups whose cycle inputs are already in device memory (mppi_optimize_group_device): the members' records are
built on the device (record_batch_kernel + path_tables_batch_kernel) from CUDA tensors, and every output is bit for bit
what mppi_optimize_batch returns for the same inputs from host memory: control sequences, fail flags, furthest points,
total and per-critic costs, cell indices, trajectories, the visualisation lattice, and the record itself byte for byte.
Also: the oracle's bars, PathAngle's undecided band, the rejections, a path_size that only the device sees, and the new
call interleaved with mppi_optimize_batch and single-handle calls.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from mpcholonavigation_b200 import abi, optimize_group_device, scenarios
from mpcholonavigation_b200.api import Engine

pytestmark = pytest.mark.gpu

RTOL, ATOL, COST_ATOL = 1e-4, 1e-6, 2e-6
MIXED_SHAPES = [(512, 56), (256, 40), (1024, 56), (384, 80)]


def _engine(fns, sc, outputs=(True, True, True), vis=False, device_map=True, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*sc.noise())
    if any(outputs):
        e.set_outputs(*outputs)
    if vis:
        e.set_visualization(5, 3)
    if device_map:
        e.set_costmap_residency(True)
    return e


def _bind(fns, engines):
    hs = (abi.H * len(engines))(*[e.h for e in engines])
    assert fns["batch_bind"](hs, len(engines)) == 0, fns["last_error"](engines[0].h)
    return hs


def _dev_cycle(cycle):
    return dataclasses.replace(cycle, costmap=torch.from_numpy(np.ascontiguousarray(cycle.costmap)).cuda())


def _inputs(cycles, stride=None):
    """the group's device inputs from the members' Cycles (maps already CUDA tensors)"""
    n = len(cycles)
    stride = stride or max(len(c.path_x) for c in cycles)
    state = np.zeros((n, 8), np.float64)
    tol = np.zeros(n, np.float64)
    size = np.zeros(n, np.int32)
    path = np.zeros((n, 3, stride), np.float32)
    for i, c in enumerate(cycles):
        state[i] = [*c.pose, *c.speed, *c.goal]
        tol[i] = c.goal_checker_xy_tolerance
        size[i] = len(c.path_x)
        path[i, 0, :size[i]], path[i, 1, :size[i]], path[i, 2, :size[i]] = c.path_x, c.path_y, c.path_yaw
    maps = [(c.costmap, c.resolution, c.origin) for c in cycles]
    return [torch.from_numpy(a).cuda() for a in (state, tol, size, path)] + [maps]


def _host_batch(fns, engines, hs, cycles):
    n = len(engines)
    ins, outs, keep, arrs = (abi.CycleIn * n)(), (abi.CycleOut * n)(), [], []
    for i, (e, c) in enumerate(zip(engines, cycles)):
        ins[i], k = c.pack()
        keep.append(k)
        outs[i], a = e._out()
        arrs.append(a)
    assert fns["optimize_batch"](hs, ins, outs, n) == 0, fns["last_error"](engines[0].h)
    return [Engine._result(outs[i], arrs[i]) for i in range(n)]


def _record(e):
    buf = np.zeros(64 * 1024, np.uint8)
    nbytes, band = C.c_uint64(0), C.c_uint64(0)
    e._check(e.f["debug_get_record"](e.h, buf.ctypes.data, buf.nbytes, C.byref(nbytes), C.byref(band)))
    return buf[:nbytes.value].copy(), band.value


def _same(a, b, ra, rb, label, full=True):
    for name in ("vx", "vy", "wz"):
        assert np.array_equal(getattr(ra, name), getattr(rb, name)), f"{label}: control {name}"
    assert ra.fail_flag == rb.fail_flag, label
    assert ra.furthest_reached_path_point == rb.furthest_reached_path_point, label
    assert np.array_equal(a.get_costs(), b.get_costs()), f"{label}: costs"
    if not full:
        return
    assert np.array_equal(a.get_cells(), b.get_cells()), f"{label}: cells"
    for q in range(a.n_critics):
        assert np.array_equal(a.get_critic_costs(q), b.get_critic_costs(q)), f"{label}: critic {q}"
    for x, y in zip(a.get_trajectories(), b.get_trajectories()):
        assert np.array_equal(x, y), f"{label}: trajectories"
    if getattr(a, "_vis", None):
        for x, y in zip(a.get_visualization(), b.get_visualization()):
            assert np.array_equal(x, y), f"{label}: visualisation"
    ka, _ = _record(a)
    kb, band = _record(b)
    assert ka.shape == kb.shape and np.array_equal(ka, kb), f"{label}: record bytes {np.flatnonzero(ka != kb)[:16]}"
    assert band == 0, f"{label}: PathAngle band hits"


# ------------------------------------------------------------------------------------------------
# scenarios: (members, path_stride or None, members whose getters and records are compared)
# ------------------------------------------------------------------------------------------------
def _near_goal(sc):
    x, y, yaw = sc.cycle.pose
    sc.cycle = dataclasses.replace(sc.cycle, goal=(x + 0.2, y + 0.05))   # Goal / GoalAngle on, the others gated off
    return sc


def _angle_open(sc):
    x, y, yaw = sc.cycle.pose
    sc.cycle = dataclasses.replace(sc.cycle, pose=(x, y, yaw + 2.0))    # the path lies 2 rad off the heading
    return sc


def _track_unknown(sc):
    sc.robot.track_unknown = 1
    cm = sc.cycle.costmap.copy()
    for k in (3, 4, 5, 12, 20):
        cm[int(sc.cycle.path_y[k] / sc.cycle.resolution), int(sc.cycle.path_x[k] / sc.cycle.resolution)] = 255
    sc.cycle = dataclasses.replace(sc.cycle, costmap=cm)
    return sc


def _path_of(sc, n):
    x, y, yaw = sc.cycle.pose
    px, py, pyaw = scenarios.straight_path(x, y, yaw, n, 2.0 / max(n - 1, 1))
    sc.cycle = dataclasses.replace(sc.cycle, path_x=px, path_y=py, path_yaw=pyaw, goal=(float(px[-1]), float(py[-1])))
    return sc


CASES = {
    "config5_two_chunks": lambda: ([scenarios.config5_robot(r, batch=512) for r in range(70)], None, (0, 33, 69)),
    "mixed_shapes": lambda: ([scenarios.config5_robot(r, batch=MIXED_SHAPES[r % 4][0], steps=MIXED_SHAPES[r % 4][1])
                              for r in range(70)], None, (0, 1, 2, 3, 69)),
    "iteration_count_2_regenerate": lambda: ([scenarios.config5_robot(r, batch=512) for r in range(6)], None, (0, 1)),
    "near_goal": lambda: ([_near_goal(scenarios.config5_robot(r, batch=512)) for r in range(6)], None, (0, 5)),
    "path_angle_open": lambda: ([_angle_open(scenarios.config5_robot(r, batch=512)) for r in range(6)], None, (0, 5)),
    "track_unknown": lambda: ([_track_unknown(scenarios.config5_robot(r, batch=512)) for r in range(6)], None, (0, 5)),
    "path_sizes": lambda: ([_path_of(scenarios.config5_robot(r, batch=512), n) for r, n in enumerate((1, 2, 40, 1024, 40, 1024))],
                           1100, (0, 1, 2, 3)),
}


@pytest.mark.parametrize("case", list(CASES))
def test_device_inputs_match_host_inputs(product_fns, oracle_fns, case):
    scs, stride, check = CASES[case]()
    n = len(scs)
    kw = [{} for _ in scs]
    outputs = (True, True, True)
    if case == "iteration_count_2_regenerate":
        kw = [dict(iteration_count=2, regenerate_noises=int(i % 2 == 1), seed=11 + i) for i in range(n)]
    if case == "path_angle_open":
        outputs = (False, True, True)   # the trajectories are spilled because PathAngle's gate is open, not on request
    host = [_engine(product_fns, sc, outputs, vis=case == "config5_two_chunks", **k) for sc, k in zip(scs, kw)]
    dev = [_engine(product_fns, sc, outputs, vis=case == "config5_two_chunks", **k) for sc, k in zip(scs, kw)]
    hh, _ = _bind(product_fns, host), _bind(product_fns, dev)
    cycles = [_dev_cycle(sc.cycle) for sc in scs]
    inputs = _inputs(cycles, stride)
    oracle_ids = (0, n - 1) if case == "config5_two_chunks" else ()
    orc = {i: _engine(oracle_fns, scs[i], device_map=False) for i in oracle_ids}
    for cycle in range(3):
        rh = _host_batch(product_fns, host, hh, cycles)
        rd = optimize_group_device(dev, *inputs)
        for i in range(n):
            _same(host[i], dev[i], rh[i], rd[i], f"{case} cycle {cycle} robot {i}", full=i in check)
        for i in oracle_ids:
            g, o = dev[i], orc[i]
            ro = o.optimize(scs[i].cycle)
            assert np.array_equal(g.get_cells(), o.get_cells()), f"robot {i}: cells vs oracle"
            np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=COST_ATOL)
            for name in ("vx", "vy", "wz"):
                np.testing.assert_allclose(getattr(rd[i], name), getattr(ro, name), rtol=RTOL, atol=ATOL)
            assert rd[i].furthest_reached_path_point == ro.furthest_reached_path_point
            o.set_control_sequence(rd[i].vx, rd[i].vy, rd[i].wz)
    if case == "iteration_count_2_regenerate":
        for i in range(n):
            for a, b in zip(host[i].get_noise(), dev[i].get_noise()):
                assert np.array_equal(a, b), f"robot {i}: noise"
    for e in host + dev + list(orc.values()):
        e.close()


def test_path_angle_band_is_counted(product_fns):
    """A path point placed on PathAngle's threshold (max_angle_to_furthest = 1 rad from the heading) is decided by the
    device's atan2f and counted; the members without such a point count nothing."""
    scs = [scenarios.config5_robot(r, batch=256) for r in range(3)]
    x, y, yaw = scs[1].cycle.pose
    px, py, pyaw = (a.copy() for a in (scs[1].cycle.path_x, scs[1].cycle.path_y, scs[1].cycle.path_yaw))
    px[10], py[10] = np.float32(x + 0.5 * np.cos(yaw + 1.0)), np.float32(y + 0.5 * np.sin(yaw + 1.0))
    scs[1].cycle = dataclasses.replace(scs[1].cycle, path_x=px, path_y=py, path_yaw=pyaw)
    dev = [_engine(product_fns, sc) for sc in scs]
    _bind(product_fns, dev)
    inputs = _inputs([_dev_cycle(sc.cycle) for sc in scs])
    optimize_group_device(dev, *inputs)
    bands = [_record(e)[1] for e in dev]
    assert bands[1] >= 1 and bands[0] == 0 and bands[2] == 0, bands
    for e in dev:
        e.close()


# ------------------------------------------------------------------------------------------------
# rejections
# ------------------------------------------------------------------------------------------------
def _launches(engines):
    return sum(e.get_profile()["kernel_launches"] for e in engines)


def _raw_call(fns, hs, n, inputs, override=None):
    state, tol, size, path, maps = inputs
    gi = abi.GroupInputs()
    gi.state, gi.goal_checker_xy_tolerance, gi.path_size, gi.path = (t.data_ptr() for t in (state, tol, size, path))
    gi.path_stride = path.shape[2]
    for k, v in (override or {}).items():
        setattr(gi, k, v)
    cms = (abi.Costmap * n)()
    for i, (cells, res, origin) in enumerate(maps[:n]):
        cms[i].cells = C.cast(C.c_void_p(cells.data_ptr()), abi.u8p)
        cms[i].size_y, cms[i].size_x = cells.shape
        cms[i].resolution = res
        cms[i].origin_x, cms[i].origin_y = origin
    outs = (abi.CycleOut * n)()
    torch.cuda.synchronize()
    return fns["optimize_group_device"](hs, n, C.byref(gi), cms, outs)


def test_rejections_enqueue_nothing(product_fns):
    n = 3
    scs = [scenarios.config5_robot(r, batch=256) for r in range(n)]
    es = [_engine(product_fns, sc, (False, False, False)) for sc in scs]
    hs = _bind(product_fns, es)
    cycles = [_dev_cycle(sc.cycle) for sc in scs]
    inputs = _inputs(cycles)
    def rejected(call, needle, first=0, restore=None):
        before = _launches(es)
        assert call() == abi.MPPI_E_CONFIG
        err = product_fns["last_error"](es[first].h).decode()   # the error is reported on the call's first handle
        assert needle in err, err
        assert _launches(es) == before, "something was launched"
        if restore:
            restore()
        # the next valid call is still correct: it matches the host-input twin below
        assert _raw_call(product_fns, hs, n, inputs) == 0, product_fns["last_error"](es[0].h)

    rejected(lambda: _raw_call(product_fns, (abi.H * n)(*[e.h for e in reversed(es)]), n, inputs), "bound group", first=n - 1)
    rejected(lambda: _raw_call(product_fns, hs, n - 1, inputs), "bound group")
    host_state = torch.zeros((n, 8), dtype=torch.float64)
    rejected(lambda: _raw_call(product_fns, hs, n, inputs, {"state": host_state.data_ptr()}), "host memory")
    pinned = torch.zeros(n, dtype=torch.int32).pin_memory()
    rejected(lambda: _raw_call(product_fns, hs, n, inputs, {"path_size": pinned.data_ptr()}), "host memory")
    # an allocation that ends before row n: the last bytes of a buffer of its own
    cudart = C.CDLL("libcudart.so.12")
    raw = C.c_void_p()
    assert cudart.cudaMalloc(C.byref(raw), C.c_size_t(1 << 21)) == 0
    try:
        short = raw.value + (1 << 21) - 8 * (n - 1)
        rejected(lambda: _raw_call(product_fns, hs, n, inputs, {"goal_checker_xy_tolerance": short}), "do not fit")
        rejected(lambda: _raw_call(product_fns, hs, n, inputs, {"path_stride": 10 ** 6}), "do not fit")
    finally:
        cudart.cudaFree(raw)
    es[2].set_profiling(True)
    rejected(lambda: _raw_call(product_fns, hs, n, inputs), "member 2", restore=lambda: es[2].set_profiling(False))
    es[1].set_costmap_residency(False)
    rejected(lambda: _raw_call(product_fns, hs, n, inputs), "host-costmap mode", restore=lambda: es[1].set_costmap_residency(True))
    # after all of that the group still computes what the host-input twin computes
    twin = [_engine(product_fns, sc, (False, False, False)) for sc in scs]
    th = _bind(product_fns, twin)
    for _ in range(8):   # as many valid device calls as the group above has made
        rt = _host_batch(product_fns, twin, th, cycles)
    rd = optimize_group_device(es, *inputs)
    rt = _host_batch(product_fns, twin, th, cycles)
    for i in range(n):
        _same(twin[i], es[i], rt[i], rd[i], f"robot {i}", full=False)
    for e in es + twin:
        e.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_inputs_on_another_device_are_rejected(product_fns):
    scs = [scenarios.config5_robot(r, batch=256) for r in range(2)]
    es = [_engine(product_fns, sc, (False, False, False)) for sc in scs]
    hs = _bind(product_fns, es)
    inputs = _inputs([_dev_cycle(sc.cycle) for sc in scs])
    other = inputs[0].to("cuda:1")
    before = _launches(es)
    assert _raw_call(product_fns, hs, 2, inputs, {"state": other.data_ptr()}) == abi.MPPI_E_CONFIG
    assert "device 1" in product_fns["last_error"](es[0].h).decode()
    assert _launches(es) == before
    for e in es:
        e.close()


def test_bad_path_size_fails_only_that_member(product_fns):
    """path_size 0 for member 1 (a regenerate_noises member): only the device sees it.  The call returns MPPI_E_CONFIG
    naming member 1, the others deliver their results, member 1's outputs are untouched, and its next cycle matches a
    twin group that never saw the bad input (control sequence, costs and noise)."""
    n = 4
    scs = [scenarios.config5_robot(r, batch=256) for r in range(n)]
    kw = [dict(regenerate_noises=int(i == 1), seed=5) for i in range(n)]
    a = [_engine(product_fns, sc, (False, False, False), **k) for sc, k in zip(scs, kw)]
    b = [_engine(product_fns, sc, (False, False, False), **k) for sc, k in zip(scs, kw)]
    _bind(product_fns, a), _bind(product_fns, b)
    good = _inputs([_dev_cycle(sc.cycle) for sc in scs])
    for engines in (a, b):
        optimize_group_device(engines, *good)
    bad = list(good)
    bad[2] = good[2].clone()
    bad[2][1] = 0
    outs = [e._out() for e in a]
    for _, arrs in outs:
        for arr in arrs:
            arr.fill(np.nan)
    hs = (abi.H * n)(*[e.h for e in a])
    state, tol, size, path, maps = bad
    gi = abi.GroupInputs()
    gi.state, gi.goal_checker_xy_tolerance, gi.path_size, gi.path = (t.data_ptr() for t in (state, tol, size, path))
    gi.path_stride = path.shape[2]
    cms = (abi.Costmap * n)()
    for i, (cells, res, origin) in enumerate(maps):
        cms[i].cells = C.cast(C.c_void_p(cells.data_ptr()), abi.u8p)
        cms[i].size_y, cms[i].size_x = cells.shape
        cms[i].resolution = res
        cms[i].origin_x, cms[i].origin_y = origin
    cout = (abi.CycleOut * n)(*[o for o, _ in outs])
    torch.cuda.synchronize()
    assert product_fns["optimize_group_device"](hs, n, C.byref(gi), cms, cout) == abi.MPPI_E_CONFIG
    assert "member 1" in product_fns["last_error"](a[0].h).decode()
    assert all(np.isnan(arr).all() for arr in outs[1][1]), "member 1's outputs were written"
    assert all(np.isfinite(arr).all() for i in (0, 2, 3) for arr in outs[i][1])
    ra, rb = optimize_group_device(a, *good), optimize_group_device(b, *good)
    _same(a[1], b[1], ra[1], rb[1], "member 1 after the bad cycle", full=False)
    for x, y in zip(a[1].get_noise(), b[1].get_noise()):
        assert np.array_equal(x, y), "member 1: noise"
    for e in a + b:
        e.close()


def test_mixed_call_sequence(product_fns, oracle_fns):
    """The new call, mppi_optimize_batch and single-handle optimize() on members of the same group, interleaved; every
    result against the oracle, so that packet tags or group state out of step would show."""
    n = 3
    scs = [scenarios.config5_robot(r, batch=512) for r in range(n)]
    es = [_engine(product_fns, sc, (False, False, False)) for sc in scs]
    hs = _bind(product_fns, es)
    orc = [_engine(oracle_fns, sc, (False, False, False), device_map=False) for sc in scs]
    cycles = [_dev_cycle(sc.cycle) for sc in scs]
    inputs = _inputs(cycles)
    for step, op in enumerate(["dev", "batch", "dev", "single", "dev", "dev", "batch", "single", "dev"]):
        if op == "dev":
            rs = optimize_group_device(es, *inputs)
        elif op == "batch":
            rs = _host_batch(product_fns, es, hs, cycles)
        else:
            rs = [es[0].optimize(cycles[0])] + [None] * (n - 1)
        for i, r in enumerate(rs):
            if r is None:
                continue
            ro = orc[i].optimize(scs[i].cycle)
            for name in ("vx", "vy", "wz"):
                np.testing.assert_allclose(getattr(r, name), getattr(ro, name), rtol=RTOL, atol=ATOL,
                                           err_msg=f"step {step} {op} robot {i} {name}")
            assert r.furthest_reached_path_point == ro.furthest_reached_path_point
            np.testing.assert_allclose(es[i].get_costs(), orc[i].get_costs(), rtol=RTOL, atol=COST_ATOL)
            es[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    for e in es + orc:
        e.close()

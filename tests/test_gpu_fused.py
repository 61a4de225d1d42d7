"""The fused small-batch kernel (tile_fused_kernel: K2 + exchange 1 + K3 + merge in one cooperative launch, zero-copy
upload, result packets in pinned host memory) against the CPU oracle and against the two-kernel path it replaces.

The parity suite (test_gpu_parity.py) already runs through the fused kernel wherever it applies (single rank, tile
layout); these cases pin what is specific to it: the exact instances (no outputs requested), the in-GPU packet
exchanges with more than 32 tiles, path sizes that change from cycle to cycle (captured graph must survive), paths
longer than the block, the zero-copy upload, multi-iteration launches, and optimize_resident after a zero-copy cycle.
"""
import dataclasses

import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, scenarios

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-6


def _engine(fns, sc, noise, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*noise)
    return e


def _close(ra, rb, rtol=RTOL, atol=ATOL, label=""):
    for name in ("vx", "vy", "wz"):
        np.testing.assert_allclose(getattr(ra, name), getattr(rb, name), rtol=rtol, atol=atol, err_msg=f"{label} {name}")
    assert ra.fail_flag == rb.fail_flag, label
    assert ra.furthest_reached_path_point == rb.furthest_reached_path_point, label


@pytest.mark.parametrize("batch,steps", [(1000, 56), (2016, 56), (4100, 33), (1000, 100), (37, 56)])
def test_exact_instance_against_oracle_and_two_kernel_path(product_fns, oracle_fns, monkeypatch, batch, steps):
    """No outputs requested -> the exact feature-set instance runs (what bench.py times).  1000: 32 tiles (one record
    per lane in the merge), 2016 / 4100: 63 / 129 tiles (general merge), 37: a ragged second tile.  Free running for 12
    cycles: fused == two-kernel path == oracle within the control tolerance, costs of all trajectories included."""
    sc = scenarios.config1(batch=batch, steps=steps)
    noise = sc.noise()
    fused = _engine(product_fns, sc, noise)
    monkeypatch.setenv("MPPI_FUSED", "0")
    two = _engine(product_fns, sc, noise)
    monkeypatch.delenv("MPPI_FUSED")
    orc = _engine(oracle_fns, sc, noise)
    for cycle in range(12):
        rf, rt, ro = fused.optimize(sc.cycle), two.optimize(sc.cycle), orc.optimize(sc.cycle)
        _close(rf, ro, label=f"fused vs oracle, cycle {cycle}")
        _close(rf, rt, label=f"fused vs two-kernel, cycle {cycle}")
        np.testing.assert_allclose(fused.get_costs(), orc.get_costs(), rtol=RTOL, atol=5e-6)
        np.testing.assert_allclose(fused.get_costs(), two.get_costs(), rtol=RTOL, atol=5e-6)
        for e in (fused, two):
            e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    assert fused.get_profile()["kernel_launches"] < two.get_profile()["kernel_launches"]   # 1 launch per cycle, not 2
    for e in (fused, two, orc):
        e.close()


def test_path_size_changes_between_cycles(product_fns, oracle_fns):
    """The pruned path changes length every cycle.  Within a 64-point bucket the captured graph is replayed (the path
    size comes from the record, not from a kernel argument); 300 points: longer than the block (loop path)."""
    sc = scenarios.config1()
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    pose = sc.cycle.pose
    for n_path in (40, 37, 52, 64, 65, 120, 300, 41, 2, 40):
        px, py, pyaw = scenarios.straight_path(pose[0], pose[1], 0.0, n_path, 0.05 if n_path < 100 else 0.008)
        cyc = dataclasses.replace(sc.cycle, path_x=px, path_y=py, path_yaw=pyaw, goal=(float(px[-1]), float(py[-1])))
        rg, ro = g.optimize(cyc), o.optimize(cyc)
        _close(rg, ro, label=f"N={n_path}")
        np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=5e-6, err_msg=f"N={n_path}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    g.close(); o.close()


def test_zero_copy_upload_is_bitwise_the_copy_engine_path(product_fns, monkeypatch):
    """record + costmap pulled out of pinned staging by the kernel itself vs one cudaMemcpyAsync: identical bits;
    and the device copies the zero-copy cycle leaves behind are complete (optimize_resident reproduces the cycle)."""
    sc = scenarios.config1()
    noise = sc.noise()
    zc = _engine(product_fns, sc, noise)
    monkeypatch.setenv("MPPI_ZERO_COPY", "0")
    cp = _engine(product_fns, sc, noise)
    monkeypatch.delenv("MPPI_ZERO_COPY")
    for cycle in range(6):
        ra, rb = zc.optimize(sc.cycle), cp.optimize(sc.cycle)
        for name in ("vx", "vy", "wz"):
            assert np.array_equal(getattr(ra, name), getattr(rb, name)), f"cycle {cycle} {name}"
        assert np.array_equal(zc.get_costs(), cp.get_costs())
    assert zc.get_profile()["h2d_bytes"] > 0
    # same warm start, resident inputs: the record and the costmap the tiles copied into device memory are all there
    before = zc.get_control_sequence()
    r1 = zc.optimize(sc.cycle)
    zc.set_control_sequence(*before)
    r2 = zc.optimize_resident()
    for name in ("vx", "vy", "wz"):
        assert np.array_equal(getattr(r1, name), getattr(r2, name)), name
    zc.close(); cp.close()


def test_timing_off_and_multi_iteration(product_fns, oracle_fns):
    """mppi_set_timing(0): no events, device_ms reads 0, same result; iteration_count = 3: three fused launches whose
    costs and furthest point carry over (optimizer.cpp:157-164), result packets only from the last one."""
    sc = scenarios.config1()
    sc.cfg["iteration_count"] = 3
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    g.set_timing(False)
    for cycle in range(5):
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        assert rg.device_ms == 0.0
        _close(rg, ro, label=f"cycle {cycle}")
        np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=3e-5)
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    g.set_timing(True)
    assert g.optimize(sc.cycle).device_ms > 0.0
    g.close(); o.close()


def test_costmap_resize_and_large_costmap_fall_back_to_the_copy_engine(product_fns, oracle_fns):
    """100x100 (zero-copy) -> 400x400 (160 KB: above the zero-copy bound, copy engine; staging buffers regrow) -> back"""
    noise = None
    g = o = None
    for map_size in (100, 400, 100):
        sc = scenarios.config1(map_size=map_size, pose=(2.5, 2.5, 0.0))
        if g is None:
            noise = sc.noise()
            g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
        for cycle in range(3):
            rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
            _close(rg, ro, label=f"map {map_size} cycle {cycle}")
            g.set_control_sequence(ro.vx, ro.vy, ro.wz)
    g.close(); o.close()


@pytest.mark.parametrize("mode", ["stream"])
def test_bound_group_against_the_single_calls(product_fns, oracle_fns, mode):
    """mppi_batch_bind: the members move to the stream layout, one strided upload and FOUR launches serve all robots;
    same controls as one mppi_optimize per robot within the tolerance (different summation order).  A member keeps
    working on its own afterwards, and the group dissolves when a member is destroyed."""
    import ctypes as C
    from mpcholonavigation_b200 import abi
    n = 9
    scs = [scenarios.config5_robot(r, batch=700) for r in range(n)]   # 22 tiles each: 198 blocks in one launch
    T = scs[0].cfg["time_steps"]
    single = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    orc = _engine(oracle_fns, scs[4], scs[4].noise())
    hs = (abi.H * n)(*[e.h for e in group])
    assert product_fns["batch_bind"](hs, n) == 0
    ins = (abi.CycleIn * n)()
    outs = (abi.CycleOut * n)()
    keep, bufs = [], []
    for i, sc in enumerate(scs):
        cin, k = sc.cycle.pack()
        ins[i] = cin
        arrs = [np.empty(T, np.float32) for _ in range(3)]
        outs[i].control_vx, outs[i].control_vy, outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
        keep.append(k); bufs.append(arrs)
    launches0 = sum(e.get_profile()["kernel_launches"] for e in group)
    for cycle in range(6):
        refs = [e.optimize(sc.cycle) for e, sc in zip(single, scs)]
        ro = orc.optimize(scs[4].cycle)
        call = product_fns["optimize_batch"] if cycle % 2 == 0 else None
        if call is not None:
            assert call(hs, ins, outs, n) == 0
        else:
            for e, sc in zip(group, scs):
                e.upload_cycle(sc.cycle)
            assert product_fns["optimize_batch_resident"](hs, outs, n) == 0
        for i in range(n):
            for a, name in zip(bufs[i], ("vx", "vy", "wz")):
                np.testing.assert_allclose(a, getattr(refs[i], name), rtol=RTOL, atol=ATOL, err_msg=f"cycle {cycle} robot {i} {name}")
            assert outs[i].fail_flag == refs[i].fail_flag
            assert outs[i].furthest_reached_path_point == refs[i].furthest_reached_path_point
        # keep both sides on the same warm start so that the comparison stays point-wise
        for i, e in enumerate(group):
            e.set_control_sequence(refs[i].vx, refs[i].vy, refs[i].wz)
        np.testing.assert_allclose(bufs[4][0], ro.vx, rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(bufs[4][2], ro.wz, rtol=RTOL, atol=ATOL)
        orc.set_control_sequence(*[b.copy() for b in bufs[4]])
    n_launches = sum(e.get_profile()["kernel_launches"] for e in group) - launches0
    assert n_launches == 24   # per cycle: four launches for 9 robots
    # a bound member on its own (shares the leader's stream), then the group again, then without the leader
    r_alone = group[3].optimize(scs[3].cycle)
    r_ref = single[3].optimize(scs[3].cycle)
    np.testing.assert_allclose(r_alone.vx, r_ref.vx, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(r_alone.wz, r_ref.wz, rtol=RTOL, atol=ATOL)
    group[0].close()                                     # dissolves the group
    group[5].set_control_sequence(*single[5].get_control_sequence())
    r_after = group[5].optimize(scs[5].cycle)
    r_ref5 = single[5].optimize(scs[5].cycle)
    np.testing.assert_allclose(r_after.vx, r_ref5.vx, rtol=RTOL, atol=ATOL)
    for e in single + group[1:] + [orc]:
        e.close()


@pytest.mark.parametrize("batch", [1000, 16384])
def test_registered_costmap_memory_is_uploaded_in_place(product_fns, batch):
    """mppi_register_costmap_memory (SURVEY 8f-4, Costmap2D::getCharMap() handed over without a staging memcpy): a
    400 x 400 costmap (160 KB, above the fused kernel's own upload bound) inside registered memory gives the same bits
    as the staged copy, in the tile layout (fused kernel behind a copy) and in the stream layout; changing the map in
    place is seen by the next cycle; unregistering falls back to staging."""
    sc = scenarios.config3(batch=batch)
    noise = sc.noise()
    a, b = _engine(product_fns, sc, noise), _engine(product_fns, sc, noise)
    cm = np.ascontiguousarray(sc.cycle.costmap)
    cyc = dataclasses.replace(sc.cycle, costmap=cm)
    b.register_costmap_memory(cm)
    for cycle in range(4):
        if cycle == 2:
            cm[180:220, 230:260] = 254          # the world changed: same buffer, new content
        ra, rb = a.optimize(cyc), b.optimize(cyc)
        for name in ("vx", "vy", "wz"):
            assert np.array_equal(getattr(ra, name), getattr(rb, name)), f"cycle {cycle} {name}"
        assert np.array_equal(a.get_costs(), b.get_costs())
        assert ra.fail_flag == rb.fail_flag
    b.unregister_costmap_memory(cm)
    ra, rb = a.optimize(cyc), b.optimize(cyc)
    assert np.array_equal(ra.vx, rb.vx) and np.array_equal(ra.wz, rb.wz)
    a.close(); b.close()


def test_mixed_call_sequence_keeps_the_packet_tags_in_step(product_fns, oracle_fns):
    """A long random mix of the entry points on ONE handle (optimize, evalControl with / without shift, resident cycles,
    speed limits, resets, explicit shifts, moving robot): every call delivers its result through the packet path, so a
    tag / epoch that got out of step would show up as a time-out or as a stale sequence.  Oracle after every call."""
    sc = scenarios.config1(batch=500)
    noise = sc.noise()
    g, o = _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    rng = np.random.default_rng(7)
    pose0 = sc.cycle.pose
    for step in range(80):
        op = rng.integers(0, 8)
        dx = float(rng.uniform(-0.05, 0.25))
        cyc = dataclasses.replace(sc.cycle, pose=(pose0[0] + dx, pose0[1] + float(rng.uniform(-0.03, 0.03)), float(rng.uniform(-0.3, 0.3))),
                                  speed=(float(rng.uniform(0, 0.3)), 0.0, float(rng.uniform(-0.2, 0.2))))
        if op <= 1:
            rg, ro = g.optimize(cyc), o.optimize(cyc)
        elif op <= 4:
            shift = bool(op % 2)
            (cg, rg), (co, ro) = g.eval_control(cyc, shift), o.eval_control(cyc, shift)
            np.testing.assert_allclose(cg, co, rtol=RTOL, atol=ATOL, err_msg=f"step {step}: command")
        elif op == 5:
            g.upload_cycle(cyc)
            rg, ro = g.optimize_resident(), o.optimize(cyc)
        elif op == 6:
            lim = float(rng.uniform(30, 100))
            g.set_speed_limit(lim, True); o.set_speed_limit(lim, True)
            rg, ro = g.optimize(cyc), o.optimize(cyc)
        else:
            g.reset(); o.reset()
            g.set_noise(*noise); o.set_noise(*noise)   # reset redraws the noise: put the shared set back
            rg, ro = g.optimize(cyc), o.optimize(cyc)
        _close(rg, ro, label=f"step {step} op {op}")
        g.set_control_sequence(ro.vx, ro.vy, ro.wz)
        g.set_control_history(o.get_control_history())
    g.close(); o.close()


@pytest.mark.parametrize("batch,steps", [(1000, 56), (2000, 56), (96, 100)])
def test_fused_kernel_is_deterministic(product_fns, batch, steps):
    """The same cycle from the same warm start, 300 times (host buffers: zero-copy upload, packet exchanges between the
    tiles, result packets): every repetition returns the bits of the first, controls and all trajectory costs.  A race
    between tiles, or between a tile's warps in shared memory, would show up as a repetition that differs."""
    sc = scenarios.config1(batch=batch, steps=steps)
    e = _engine(product_fns, sc, sc.noise())
    for _ in range(5):                       # a non-trivial warm start
        e.optimize(sc.cycle)
    start = e.get_control_sequence()
    ref = None
    for rep in range(300):
        e.set_control_sequence(*start)
        r = e.optimize(sc.cycle)
        got = (r.vx.copy(), r.vy.copy(), r.wz.copy(), e.get_costs() if rep % 25 == 0 else None, r.fail_flag,
               r.furthest_reached_path_point)
        if ref is None:
            ref = got
            continue
        for a, b in zip(got[:3], ref[:3]):
            assert np.array_equal(a, b), f"repetition {rep} differs"
        if got[3] is not None:
            assert np.array_equal(got[3], ref[3]), f"repetition {rep}: costs differ"
        assert got[4:] == ref[4:]
    e.close()


def test_boxed_in_footprint_branch_through_the_fused_kernel(product_fns, oracle_fns):
    """configs[1] with the robot boxed in (rectangular footprint inside a ring of discs, scenarios.config1(ring=0.47)): CostCritic
    takes the footprint branch (cost_critic.cpp:204-209) for more than a tenth of the visited poses in every cycle.  Exact
    instance (what bench-style calls run) and the instance with outputs: cells and trajectories bit-equal, costs and controls
    at the usual bars."""
    import ctypes as C
    sc = scenarios.config1(footprint="rectangle", ring=0.47)
    noise = sc.noise()
    exact, full, orc = _engine(product_fns, sc, noise), _engine(product_fns, sc, noise), _engine(oracle_fns, sc, noise)
    for e in (full, orc):
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    counters = (C.c_uint64 * 4)()
    for cycle in range(6):
        re_, rf, ro = exact.optimize(sc.cycle), full.optimize(sc.cycle), orc.optimize(sc.cycle)
        _close(re_, ro, label=f"exact instance, cycle {cycle}")
        _close(rf, ro, label=f"instance with outputs, cycle {cycle}")
        assert np.array_equal(full.get_cells(), orc.get_cells())
        for a, b in zip(full.get_trajectories(), orc.get_trajectories()):
            assert np.array_equal(a, b)
        for e in (exact, full):
            np.testing.assert_allclose(e.get_costs(), orc.get_costs(), rtol=RTOL, atol=5e-6)
            e.set_control_sequence(ro.vx, ro.vy, ro.wz)
        oracle_fns["get_counters"](orc.h, counters)
        assert counters[1] > 0.08 * counters[0] > 0, list(counters)
    for e in (exact, full, orc):
        e.close()

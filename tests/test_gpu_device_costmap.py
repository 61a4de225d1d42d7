"""Device-resident costmaps (mppi_set_costmap_residency(MPPI_COSTMAP_DEVICE)): the same cycle with the map in host memory
and with the same bytes in a CUDA torch tensor gives the same bits on every path (control sequence, fail_flag, furthest
point, total and per-critic costs, cell indices), and stays within the oracle's bars.  The device run makes the
path-validity tables on the device (path_tables_kernel); the host run makes them in build_params.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from mpcholonavigation_b200 import Engine, MppiError, abi, optimize_sharded, scenarios, sharding

pytestmark = pytest.mark.gpu

RTOL, ATOL, COST_ATOL = 1e-4, 1e-6, 2e-6


def _engine(fns, sc, noise=None, outputs=True, device_map=False, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise is not None:
        e.set_noise(*noise)
    if outputs:
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    if device_map:
        e.set_costmap_residency(True)
    return e


def _on_device(cycle):
    return dataclasses.replace(cycle, costmap=torch.from_numpy(np.ascontiguousarray(cycle.costmap)).cuda())


def _same(eh, ed, rh, rd, n_critics, label, outputs=True):
    """host-map run == device-map run, bit for bit"""
    for name in ("vx", "vy", "wz"):
        assert np.array_equal(getattr(rh, name), getattr(rd, name)), f"{label}: control {name}"
    assert rh.fail_flag == rd.fail_flag, label
    assert rh.furthest_reached_path_point == rd.furthest_reached_path_point, label
    assert np.array_equal(eh.get_costs(), ed.get_costs()), f"{label}: costs"
    if outputs:
        assert np.array_equal(eh.get_cells(), ed.get_cells()), f"{label}: cells"
        for q in range(n_critics):
            assert np.array_equal(eh.get_critic_costs(q), ed.get_critic_costs(q)), f"{label}: critic {q}"


def _oracle_bars(g, o, rg, ro, n_critics, label, outputs=True, cost_atol=COST_ATOL):
    if outputs:
        assert np.array_equal(g.get_cells(), o.get_cells()), f"{label}: cells vs oracle"
        for q in range(n_critics):
            np.testing.assert_allclose(g.get_critic_costs(q), o.get_critic_costs(q), rtol=RTOL, atol=COST_ATOL,
                                       err_msg=f"{label}: critic {q} vs oracle")
    np.testing.assert_allclose(g.get_costs(), o.get_costs(), rtol=RTOL, atol=cost_atol, err_msg=f"{label}: costs vs oracle")
    for name in ("vx", "vy", "wz"):
        np.testing.assert_allclose(getattr(rg, name), getattr(ro, name), rtol=RTOL, atol=ATOL, err_msg=f"{label}: {name} vs oracle")
    assert bool(rg.fail_flag) == bool(ro.fail_flag), label
    assert rg.furthest_reached_path_point == ro.furthest_reached_path_point, label


PATHS = {
    # name: (scenario, config overrides, environment, call)
    "fused": (lambda: scenarios.config1(), {}, {}, "optimize"),
    "fused_exact_instance": (lambda: scenarios.config1(), {}, {}, "optimize_no_outputs"),
    "two_kernel_tile": (lambda: scenarios.config1(), {}, {"MPPI_FUSED": "0"}, "optimize"),
    "stream_footprint": (lambda: scenarios.config3(), {}, {}, "optimize"),
    "stream_boxed_in": (lambda: scenarios.config3(dense=True), {}, {}, "optimize"),
    "iteration_count_2": (lambda: scenarios.config1(), {"iteration_count": 2}, {}, "optimize"),
    "eval_control": (lambda: scenarios.config1(), {}, {}, "eval_control"),
    "upload_resident": (lambda: scenarios.config1(), {}, {}, "resident"),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_device_map_matches_host_map(product_fns, oracle_fns, monkeypatch, path):
    make, over, env, call = PATHS[path]
    sc = make()
    sc.cfg.update(over)
    noise = sc.noise()
    outputs = call != "optimize_no_outputs"
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eh = _engine(product_fns, sc, noise, outputs)
    ed = _engine(product_fns, sc, noise, outputs, device_map=True)
    for k in env:
        monkeypatch.delenv(k)
    o = _engine(oracle_fns, sc, noise)
    dev_cycle = _on_device(sc.cycle)
    n_crit = len(sc.critics)
    for cycle in range(3):
        if call == "eval_control":
            ch, rh = eh.eval_control(sc.cycle, True)
            cd, rd = ed.eval_control(dev_cycle, True)
            assert np.array_equal(ch, cd), f"cycle {cycle}: command"
            assert np.array_equal(eh.get_control_history(), ed.get_control_history())
        elif call == "resident":
            eh.upload_cycle(sc.cycle)
            ed.upload_cycle(dev_cycle)
            rh, rd = eh.optimize_resident(), ed.optimize_resident()
        else:
            rh, rd = eh.optimize(sc.cycle), ed.optimize(dev_cycle)
        _same(eh, ed, rh, rd, n_crit, f"{path} cycle {cycle}", outputs)
        ro = o.optimize(sc.cycle)
        if "iteration_count" in over:
            # the oracle's second iteration starts from its own first update: the bars of the multi-iteration tests
            _oracle_bars(ed, o, rd, ro, n_crit, f"{path} cycle {cycle}", outputs=False, cost_atol=3e-5)
        elif call != "eval_control":   # evalControl shifted the device sequence: the oracle comparison is optimize()'s
            _oracle_bars(ed, o, rd, ro, n_crit, f"{path} cycle {cycle}", outputs)
        for e in (eh, ed):
            e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    for e in (eh, ed, o):
        e.close()


def test_regenerate_noises(product_fns):
    """Philox noise redrawn behind every result: the redraw does not read the map, both handles draw the same sets"""
    sc = scenarios.config1()
    eh = _engine(product_fns, sc, regenerate_noises=1, seed=7)
    ed = _engine(product_fns, sc, device_map=True, regenerate_noises=1, seed=7)
    dev_cycle = _on_device(sc.cycle)
    for cycle in range(5):
        rh, rd = eh.optimize(sc.cycle), ed.optimize(dev_cycle)
        _same(eh, ed, rh, rd, len(sc.critics), f"cycle {cycle}")
    eh.close(); ed.close()


def test_sharded_two_handles_one_gpu(product_fns, oracle_fns):
    sc = scenarios.config1(batch=1024)
    noise = sc.noise()
    B = sc.cfg["batch_size"]

    def shards(device_map):
        es = []
        for r in range(2):
            b0, b1 = sharding.shard_bounds(B, r, 2)
            e = _engine(product_fns, sc, [p[b0:b1] for p in noise], outputs=False, device_map=device_map,
                        batch_size=b1 - b0, shard_offset=b0, shard_total=B)
            es.append(e)
        return es

    sh, sd = shards(False), shards(True)
    o = _engine(oracle_fns, sc, noise, outputs=False)
    dev_cycle = _on_device(sc.cycle)
    for cycle in range(3):
        rh, rd, ro = optimize_sharded(sh, sc.cycle), optimize_sharded(sd, dev_cycle), o.optimize(sc.cycle)
        for name in ("vx", "vy", "wz"):
            assert np.array_equal(getattr(rh, name), getattr(rd, name)), f"cycle {cycle} {name}"
            np.testing.assert_allclose(getattr(rd, name), getattr(ro, name), rtol=RTOL, atol=ATOL)
        assert rh.fail_flag == rd.fail_flag and rh.furthest_reached_path_point == rd.furthest_reached_path_point
        assert rd.furthest_reached_path_point == ro.furthest_reached_path_point
        for a, b in zip(sh, sd):
            assert np.array_equal(a.get_costs(), b.get_costs())
        for e in sh + sd:
            e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    for e in sh + sd + [o]:
        e.close()


# ------------------------------------------------------------------------------------------------
# path tables: one category of invalid path point at a time, each at the edge of what flips PathAlign's occupancy gate
# ------------------------------------------------------------------------------------------------
UNKNOWN, INSCRIBED, LETHAL = 255, 253, 254
ALIGN_Q, FOLLOW_Q = 4, 5   # PathAlignCritic, PathFollowCritic in omni_default_critics
KINDS = {"unknown": (UNKNOWN, False), "unknown_tracked": (UNKNOWN, True), "inscribed": (INSCRIBED, False),
         "lethal": (LETHAL, False), "off_map": (None, False)}


def _tables_scenario(kind, marked, f=None):
    """The robot at (1.0, 2.5) heading +x on a free 5 x 5 m map; the path runs 0.5 m beside it (out of the footprint's
    reach), 80 points on consecutive cell centres of row 60.  PathAlign with offset_from_furthest 5 and
    max_path_occupancy_ratio 0.02.  Given the furthest reached point f, the points 3, 4, 5 and f + 5 are made invalid
    (marked=True) by `kind`: three invalid points among [closest = 0, f) close the gate (more than two, 3 / f > 0.02; one
    fewer would leave it open), and PathFollow's target f + 5 moves to f + 6.  Off the map: those four points sit one
    row higher, on the row the marked map no longer has (61 rows instead of 100)."""
    sc = scenarios.config1(pose=(1.0, 2.5, 0.0))
    sc.critics = [(n, dict(kw, max_path_occupancy_ratio=0.02, offset_from_furthest=5)) if n == "PathAlignCritic" else (n, kw)
                  for n, kw in sc.critics]
    res = sc.cycle.resolution
    px = (1.025 + res * np.arange(80)).astype(np.float32)
    py = np.full(80, 3.025, np.float32)
    cm = np.zeros((100, 100), np.uint8)
    value, track_unknown = KINDS[kind]
    if f is not None:
        pts = [3, 4, 5, f + 5]
        if value is None:
            py[pts] = np.float32(3.075)
            if marked:
                cm = np.ascontiguousarray(cm[:61])
        elif marked:
            for j in pts:
                cm[int(py[j] / res), int(px[j] / res)] = value
    sc.cycle = dataclasses.replace(sc.cycle, path_x=px, path_y=py, path_yaw=np.zeros(80, np.float32),
                                   goal=(float(px[-1]), float(py[-1])), costmap=cm)
    sc.robot.track_unknown = int(track_unknown)
    return sc


@pytest.mark.parametrize("kind", list(KINDS))
def test_path_tables(product_fns, oracle_fns, kind):
    probe = _tables_scenario(kind, False)
    noise = probe.noise()
    T = probe.cfg["time_steps"]
    warm = (np.full(T, 0.4, np.float32), np.zeros(T, np.float32), np.zeros(T, np.float32))
    ep = _engine(product_fns, probe, noise, outputs=False)
    ep.set_control_sequence(*warm)
    f = ep.optimize(probe.cycle).furthest_reached_path_point
    ep.close()
    assert f is not None and 6 <= f <= 70, f   # 3 / f > 0.02 and f + 6 on the path
    marked, free = _tables_scenario(kind, True, f), _tables_scenario(kind, False, f)
    eh, ed = _engine(product_fns, marked, noise), _engine(product_fns, marked, noise, device_map=True)
    ef, o = _engine(product_fns, free, noise), _engine(oracle_fns, marked, noise)
    dev_cycle = _on_device(marked.cycle)
    n_crit = len(marked.critics)
    for e in (eh, ed, ef, o):
        e.set_control_sequence(*warm)
    for cycle in range(3):
        rh, rd, rf, ro = eh.optimize(marked.cycle), ed.optimize(dev_cycle), ef.optimize(free.cycle), o.optimize(marked.cycle)
        _same(eh, ed, rh, rd, n_crit, f"{kind} cycle {cycle}")
        _oracle_bars(ed, o, rd, ro, n_crit, f"{kind} cycle {cycle}")
        if cycle == 0:
            assert rh.furthest_reached_path_point == rf.furthest_reached_path_point == f
            align_h, align_f = eh.get_critic_costs(ALIGN_Q), ef.get_critic_costs(ALIGN_Q)
            follow_h, follow_f = eh.get_critic_costs(FOLLOW_Q), ef.get_critic_costs(FOLLOW_Q)
            assert align_f.any(), "PathAlign does not run on the free map"
            if kind == "unknown_tracked":
                # unknown space is tracked: the same points are valid, the tables are the free map's
                assert np.array_equal(align_h, align_f) and np.array_equal(follow_h, follow_f)
            else:
                assert not align_h.any(), f"{kind}: PathAlign gate did not close"
                assert not np.array_equal(follow_h, follow_f), f"{kind}: PathFollow target did not move"
        for e in (eh, ed, ef, o):
            e.set_control_sequence(*warm)
    for e in (eh, ed, ef, o):
        e.close()


def test_changing_pointer_every_cycle(product_fns):
    """Two tensors with different obstacles, alternated over 12 cycles on one handle whose cycle is a replayed graph: every
    cycle matches its host twin, so no captured node keeps a stale map pointer."""
    sa, sb = scenarios.config1(map_seed=0), scenarios.config1(map_seed=5)
    assert not np.array_equal(sa.cycle.costmap, sb.cycle.costmap)
    noise = sa.noise()
    eh, ed = _engine(product_fns, sa, noise), _engine(product_fns, sa, noise, device_map=True)
    da, db = _on_device(sa.cycle), _on_device(sb.cycle)
    for cycle in range(12):
        host, dev = (sa.cycle, da) if cycle % 2 == 0 else (sb.cycle, db)
        rh, rd = eh.optimize(host), ed.optimize(dev)
        _same(eh, ed, rh, rd, len(sa.critics), f"cycle {cycle}")
    eh.close(); ed.close()


# ------------------------------------------------------------------------------------------------
# robot groups
# ------------------------------------------------------------------------------------------------
def _bind(fns, engines):
    hs = (abi.H * len(engines))(*[e.h for e in engines])
    assert fns["batch_bind"](hs, len(engines)) == 0
    return hs


def test_group_shared_private_and_host_maps(product_fns, oracle_fns):
    """70 members (two chunks): 0-29 share one 1000 x 1000 map (1 MB, more than a group slice holds), 30-59 have private
    device maps, 60-69 stay in host mode.  The same group with every map in host memory (bound after its slices were
    grown to the large map) is the twin; mppi_optimize_batch and _resident both run."""
    n, T = 70, 56
    scs = [scenarios.config5_robot(r, batch=512, steps=T) for r in range(n)]
    big = np.zeros((1000, 1000), np.uint8)
    big[:100, :100] = scs[0].cycle.costmap
    big[400:500, 300:400] = scs[1].cycle.costmap
    for i in range(30):
        scs[i].cycle = dataclasses.replace(scs[i].cycle, costmap=big)
    big_dev = torch.from_numpy(big).cuda()
    dev_cycles = [dataclasses.replace(sc.cycle, costmap=big_dev) if i < 30 else
                  (_on_device(sc.cycle) if i < 60 else sc.cycle) for i, sc in enumerate(scs)]
    host = [_engine(product_fns, sc, sc.noise(), outputs=False) for sc in scs]
    dev = [_engine(product_fns, sc, sc.noise(), outputs=False, device_map=i < 60) for i, sc in enumerate(scs)]
    host[0].upload_cycle(scs[0].cycle)   # grows its staging to the large map: the group's slices are bound at that size
    hh, hd = _bind(product_fns, host), _bind(product_fns, dev)
    ids = (0, 29, 45, 65)
    orc = {i: _engine(oracle_fns, scs[i], scs[i].noise(), outputs=False) for i in ids}

    def run(engines, hs, cycles, resident):
        outs = (abi.CycleOut * n)()
        bufs = []
        for i in range(n):
            arrs = [np.empty(T, np.float32) for _ in range(3)]
            outs[i].control_vx, outs[i].control_vy, outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
            bufs.append(arrs)
        if resident:
            for e, c in zip(engines, cycles):
                e.upload_cycle(c)
            assert product_fns["optimize_batch_resident"](hs, outs, n) == 0
        else:
            ins = (abi.CycleIn * n)()
            keep = []
            for i, c in enumerate(cycles):
                cin, k = c.pack()
                ins[i] = cin
                keep.append(k)
            assert product_fns["optimize_batch"](hs, ins, outs, n) == 0, engines[0].f["last_error"](engines[0].h)
        return outs, bufs

    for cycle in range(4):
        resident = cycle % 2 == 1
        oh, bh = run(host, hh, [sc.cycle for sc in scs], resident)
        od, bd = run(dev, hd, dev_cycles, resident)
        for i in range(n):
            for a, b, name in zip(bh[i], bd[i], ("vx", "vy", "wz")):
                assert np.array_equal(a, b), f"cycle {cycle} robot {i} {name}"
            assert oh[i].fail_flag == od[i].fail_flag, (cycle, i)
            assert oh[i].furthest_reached_path_point == od[i].furthest_reached_path_point, (cycle, i)
            assert np.array_equal(host[i].get_costs(), dev[i].get_costs()), (cycle, i)
        for i in ids:
            ro = orc[i].optimize(scs[i].cycle)
            for a, name in zip(bd[i], ("vx", "vy", "wz")):
                np.testing.assert_allclose(a, getattr(ro, name), rtol=RTOL, atol=ATOL, err_msg=f"cycle {cycle} robot {i} {name}")
            assert od[i].furthest_reached_path_point == ro.furthest_reached_path_point
            np.testing.assert_allclose(dev[i].get_costs(), orc[i].get_costs(), rtol=RTOL, atol=COST_ATOL)
            orc[i].set_control_sequence(*[b.copy() for b in bd[i]])
    for e in host + dev + list(orc.values()):
        e.close()


# ------------------------------------------------------------------------------------------------
# rejections
# ------------------------------------------------------------------------------------------------
def _status_and_launches(e, fn):
    before = e.get_profile()["kernel_launches"]
    with pytest.raises(MppiError) as err:
        fn()
    assert "status %d" % abi.MPPI_E_CONFIG in str(err.value), str(err.value)
    assert e.get_profile()["kernel_launches"] == before, "something was launched"
    return str(err.value)


def test_rejections(product_fns):
    sc = scenarios.config1(batch=256)
    noise = sc.noise()
    e = _engine(product_fns, sc, noise, device_map=True)
    msg = _status_and_launches(e, lambda: e.optimize(sc.cycle))   # numpy map in device mode
    assert "host memory" in msg
    _status_and_launches(e, lambda: e.eval_control(sc.cycle, False))
    _status_and_launches(e, lambda: e.upload_cycle(sc.cycle))
    B, T = sc.cfg["batch_size"], sc.cfg["time_steps"]
    planes = [np.zeros((B, T), np.float32) for _ in range(6)]
    _status_and_launches(e, lambda: e.score_trajectories(_on_device(sc.cycle), *planes))
    # a map smaller than its geometry says: rejected before any kernel sees it
    short = dataclasses.replace(sc.cycle, costmap=torch.zeros((10, 10), dtype=torch.uint8, device="cuda"))
    cin, keep = short.pack()
    cin.costmap.size_x = cin.costmap.size_y = 4000
    out, _ = e._out()
    assert product_fns["optimize"](e.h, C.byref(cin), C.byref(out)) == abi.MPPI_E_CONFIG
    # integrate_state_velocities needs no map and keeps working
    h = _engine(product_fns, sc, noise)
    vel = [np.random.default_rng(3).standard_normal((B, T)).astype(np.float32) * 0.2 for _ in range(3)]
    for a, b in zip(e.integrate_state_velocities(sc.cycle.pose, *vel), h.integrate_state_velocities(sc.cycle.pose, *vel)):
        assert np.array_equal(a, b)
    # after the rejections the handle still runs a device-map cycle
    r = e.optimize(_on_device(sc.cycle))
    assert np.isfinite(r.vx).all()
    e.close(); h.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_map_on_another_device_is_rejected(product_fns):
    sc = scenarios.config1(batch=256)
    e = _engine(product_fns, sc, sc.noise(), device_map=True)
    other = dataclasses.replace(sc.cycle, costmap=torch.from_numpy(np.ascontiguousarray(sc.cycle.costmap)).to("cuda:1"))
    msg = _status_and_launches(e, lambda: e.optimize(other))
    assert "device 1" in msg
    e.close()


def test_rejected_upload_leaves_nothing_to_run(product_fns):
    """A device-mode mppi_upload_cycle whose map is rejected ends the resident cycle: the next mppi_optimize_resident (one
    handle) and mppi_optimize_batch_resident (a bound group) fail with MPPI_E_STATE and launch nothing - they never replay
    a record whose map pointer was rejected or whose map's call is over."""
    n, T = 3, 56
    scs = [scenarios.config5_robot(r, batch=256, steps=T) for r in range(n)]
    es = [_engine(product_fns, sc, sc.noise(), outputs=False, device_map=True) for sc in scs]
    dev_cycles = [_on_device(sc.cycle) for sc in scs]   # the maps stay alive until the resident calls return
    single = _engine(product_fns, scs[0], scs[0].noise(), outputs=False, device_map=True)
    single.upload_cycle(dev_cycles[0])
    single.optimize_resident()
    _status_and_launches(single, lambda: single.upload_cycle(scs[0].cycle))   # numpy map in device mode
    before = single.get_profile()["kernel_launches"]
    with pytest.raises(MppiError) as err:
        single.optimize_resident()
    assert "status %d" % abi.MPPI_E_STATE in str(err.value)
    assert single.get_profile()["kernel_launches"] == before
    hs = _bind(product_fns, es)
    outs = (abi.CycleOut * n)()
    for e, c in zip(es, dev_cycles):
        e.upload_cycle(c)
    assert product_fns["optimize_batch_resident"](hs, outs, n) == 0
    _status_and_launches(es[1], lambda: es[1].upload_cycle(scs[1].cycle))
    before = sum(e.get_profile()["kernel_launches"] for e in es)
    assert product_fns["optimize_batch_resident"](hs, outs, n) == abi.MPPI_E_STATE
    assert sum(e.get_profile()["kernel_launches"] for e in es) == before, "something was launched"
    # the group runs again once the member has a valid upload
    es[1].upload_cycle(dev_cycles[1])
    assert product_fns["optimize_batch_resident"](hs, outs, n) == 0
    for e in es + [single]:
        e.close()


def test_sharded_mixed_residency_is_rejected(product_fns):
    """The shards of mppi_optimize_sharded read one costmap.cells: a host-mode shard must not memcpy from a device map"""
    sc = scenarios.config1(batch=1024)
    noise = sc.noise()
    es = []
    for r in range(2):
        b0, b1 = sharding.shard_bounds(1024, r, 2)
        es.append(_engine(product_fns, sc, [p[b0:b1] for p in noise], outputs=False, device_map=r == 0,
                          batch_size=b1 - b0, shard_offset=b0, shard_total=1024))
    before = sum(e.get_profile()["kernel_launches"] for e in es)
    with pytest.raises(MppiError) as err:
        optimize_sharded(es, _on_device(sc.cycle))
    assert "residency" in str(err.value)
    assert sum(e.get_profile()["kernel_launches"] for e in es) == before
    for e in es:
        e.close()

"""Parity of the CUDA paths against the CPU oracle away from the deployed parameters (tests/param_space.py): optimizer
profiles with three distinct stds and limits, vx_min below, at and above zero, temperatures 1e-3 to 5, gamma 0 and 0.3,
Ackermann at two turning radii and DiffDrive; critic lists with cost_power 2 and 3, PathAlign steps 1 ... T + 3, the
PathAngle gate on both of its branches, disabled and permuted critics; speed limits changed between cycles; the
softmax at low temperature with its minimum in the last tile, chunk or shard; merges of more partial records than
merge_finalize_body caches; noise transposes of batches whose row blocks exceed a grid's 65535 y blocks.

Bars as in test_gpu_map_frames.py.  Beside the oracle, every cycle's controls are checked against update_fp64 of the
device's own noise, warm start and total costs, so a wrong clip or weighted sum shows even where the oracle agrees with
it.  Every test asserts the edge it is about - the (plane, side) pairs that clipped per path, the coupling, the
argmin's tile / chunk / shard, the effective sample size, the gate states - and prints it.
"""
import dataclasses

import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, abi, optimize_group_device, optimize_sharded, sharding
from tests import param_space as ps
from tests.test_gpu_group_device_inputs import _host_batch, _inputs
from tests.test_gpu_map_frames import ATOL, COST_ATOL, RTOL, _bars, _bind, _clear_env, _on_device, _set_env

pytestmark = pytest.mark.gpu

STREAM = {"MPPI_STREAM_MIN_BATCH": "1"}
# path: (batch, environment, kind)
PATHS = {
    "fused": (1000, {}, "optimize"),
    "two_kernel": (1000, {"MPPI_FUSED": "0"}, "optimize"),         # K3's last block merges and clips (finalize_controls)
    "two_kernel_2048": (2048, {"MPPI_FUSED": "0"}, "optimize"),    # 64 K3 blocks: still K3's last block (kLastBlockMergeMax)
    "two_kernel_k4": (2049, {"MPPI_FUSED": "0"}, "optimize"),      # 65 K3 blocks: merge_finalize_kernel
    "stream_tma": (1024, STREAM, "optimize"),                      # B % 4 == 0: weighted_sums_tma_kernel's own merge
    "stream_b4r1": (1025, STREAM, "optimize"),                     # B % 4 != 0: merge_finalize_kernel
    "stream_b4r2": (1026, STREAM, "optimize"),
    "stream_b4r3": (1027, STREAM, "optimize"),
    "iteration_count_2": (1000, {}, "iterations"),
    "eval_control_shift": (1000, {}, "eval_control"),
    "sharded": (1000, {}, "sharded"),
}
T = 56


def _engine(fns, sc, nz, env=None, monkeypatch=None, outputs=True, **kw):
    if env:
        _set_env(monkeypatch, env)
    e = Engine(fns, **{**sc.cfg, **kw})
    if env:
        _clear_env(monkeypatch, env)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*nz)
    if outputs:
        e.set_outputs(trajectories=True, cells=True, critic_costs=True)
    return e


def _shards(fns, sc, nz, n=2):
    B = sc.cfg["batch_size"]
    out = []
    for r in range(n):
        b0, b1 = sharding.shard_bounds(B, r, n)
        e = Engine(fns, **dict(sc.cfg, batch_size=b1 - b0, shard_offset=b0, shard_total=B))
        e.set_robot(sc.robot)
        e.set_critics(sc.critics)
        e.set_noise(*[None if a is None else a[b0:b1] for a in nz])
        out.append(e)
    return out


def _controls(r):
    return np.stack([r.vx, r.vy, r.wz])


def _fp64(label, cfg, cs, nz, totals, got, lims=None, rtol=RTOL, atol=ATOL):
    """the device's controls are update_fp64 of its own noise, warm start and total costs"""
    u = ps.update_fp64(cs, ps.noise_planes(nz, cfg), totals, dict(cfg, gamma=0.0), lims)
    np.testing.assert_allclose(got, u.controls, rtol=rtol, atol=atol, err_msg=f"{label}: controls vs update_fp64")
    return u


def _control_floor(o, cfg):
    """absolute floor of the control bar where the totals are large (cost_power 2 / 3) or the batch reductions run over
    2048 rows and more (the merge order of K3's last block and K4 against the oracle's index order): one fp32 ulp of
    the lowest total moves a softmax weight by ulp / temperature, so four of them bound what two legal summation orders
    of the same costs can put between the controls"""
    return max(ATOL, 4.0 * float(np.spacing(np.float32(o.get_costs().min()))) / cfg["temperature"])


def _want_saturated(cfg):
    return {(p, s) for p in ((0, 1, 2) if ps.holonomic(cfg) else (0, 2)) for s in (-1, 1)}


def _check_coupling(cfg, us, label):
    if cfg["motion_model"] == "Ackermann":
        assert sum(int(u.coupled.sum()) for u in us) >= 4, f"{label}: the Ackermann coupling never acted"


# ------------------------------------------------------------------------------------------------
# A. profiles x paths, every bound clipped
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("profile", list(ps.PROFILES))
def test_profile_parity(product_fns, oracle_fns, monkeypatch, profile, path):
    B, env, kind = PATHS[path]
    cfg = ps.profile_cfg(profile, B, T, iteration_count=2 if kind == "iterations" else 1)
    sc = ps.scene(cfg, seed=11)
    nz = ps.noise(cfg, 11)
    n_critics = len(sc.critics)
    o = _engine(oracle_fns, sc, nz)
    cs = ps.warm_start(cfg)
    us, seen = [], set()
    if kind == "sharded":
        shards = _shards(product_fns, sc, nz)
        for cycle in range(2):
            label = f"{profile} {path} cycle {cycle}"
            for e in shards + [o]:
                e.set_control_sequence(*cs)
            rs, ro = optimize_sharded(shards, sc.cycle), o.optimize(sc.cycle)
            totals = np.concatenate([e.get_costs() for e in shards])
            np.testing.assert_allclose(totals, o.get_costs(), rtol=RTOL, atol=COST_ATOL, err_msg=label)
            np.testing.assert_allclose(_controls(rs), _controls(ro), rtol=RTOL, atol=ATOL, err_msg=label)
            assert rs.fail_flag == ro.fail_flag and rs.furthest_reached_path_point == ro.furthest_reached_path_point
            us.append(_fp64(label, cfg, cs, nz, totals, _controls(rs)))
        for e in shards:
            e.close()
    else:
        g = _engine(product_fns, sc, nz, env, monkeypatch)
        g1 = _engine(product_fns, dataclasses.replace(sc, cfg=dict(sc.cfg, iteration_count=1)), nz) if kind == "iterations" else None
        hist = np.arange(12, dtype=np.float32).reshape(4, 3) * 0.01
        for cycle in range(2):
            label = f"{profile} {path} cycle {cycle}"
            for e in (g, o, g1):
                if e is not None:
                    e.set_control_sequence(*cs)
            if g1 is not None:
                r1 = g1.optimize(sc.cycle)
                us.append(_fp64(label + " first iteration", cfg, cs, nz, g1.get_costs(), _controls(r1)))
                pin = [np.ascontiguousarray(a, dtype=np.float32) for a in (r1.vx, r1.vy, r1.wz)]
                f32p = oracle_fns["_lib"].oracle_set_iteration_controls.argtypes[2]
                assert oracle_fns["set_iteration_controls"](o.h, 0, *[a.ctypes.data_as(f32p) for a in pin]) == 0
            if kind == "eval_control":
                for e in (g, o):
                    e.set_control_history(hist)
                cmd_g, rg = g.eval_control(sc.cycle, True)
                cmd_o, ro = o.eval_control(sc.cycle, True)
                np.testing.assert_allclose(cmd_g, cmd_o, rtol=RTOL, atol=ATOL, err_msg=f"{label}: command")
                np.testing.assert_allclose(g.get_control_history(), o.get_control_history(), rtol=RTOL, atol=ATOL)
                np.testing.assert_allclose(np.stack(g.get_control_sequence()), np.stack(o.get_control_sequence()),
                                           rtol=RTOL, atol=ATOL, err_msg=f"{label}: shifted sequence")
            else:
                rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
            atol = 1e-5 if g1 is not None else (_control_floor(o, cfg) if path in ("two_kernel_2048", "two_kernel_k4") else ATOL)
            _bars(g, o, rg, ro, n_critics, label, control_atol=atol)
            if kind == "optimize":
                us.append(_fp64(label, cfg, cs, nz, g.get_costs(), _controls(rg)))
            elif kind == "eval_control":
                # the clip ahead of the filter and the shift, counted on the device's own costs
                us.append(ps.update_fp64(cs, ps.noise_planes(nz, cfg), g.get_costs(), dict(cfg, gamma=0.0)))
            if not ps.holonomic(cfg) and kind != "eval_control":   # (evalControl returns the filtered sequence)
                assert np.array_equal(rg.vy, cs[1]), f"{label}: the lateral plane of a non-holonomic model moved"
        for e in (g, g1):
            if e is not None:
                e.close()
    o.close()
    for u in us:
        seen |= u.saturated()
    print(f"{profile} {path}: saturated (plane, side) {sorted(seen)}, coupled steps {[int(u.coupled.sum()) for u in us]}")
    assert seen == _want_saturated(cfg), f"{profile} {path}: saturated {sorted(seen)}"
    _check_coupling(cfg, us, f"{profile} {path}")


def test_group_of_profiles(product_fns, oracle_fns):
    """one bound group whose members each run another profile (and batch size): mppi_optimize_batch against each
    member's oracle and update_fp64, every member's bounds clipped"""
    names = list(ps.PROFILES)
    cfgs = [ps.profile_cfg(n, 384 + 129 * i, T) for i, n in enumerate(names)]
    scs = [ps.scene(c, seed=40 + i) for i, c in enumerate(cfgs)]
    nzs = [ps.noise(c, 40 + i) for i, c in enumerate(cfgs)]
    gs = [_engine(product_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    os_ = [_engine(oracle_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    hs = _bind(product_fns, gs)
    for cycle in range(2):
        css = [ps.warm_start(c) for c in cfgs]
        for e, f, cs in zip(gs, os_, css):
            e.set_control_sequence(*cs)
            f.set_control_sequence(*cs)
        rs = _host_batch(product_fns, gs, hs, [sc.cycle for sc in scs])
        for i, name in enumerate(names):
            label = f"member {i} ({name}) cycle {cycle}"
            ro = os_[i].optimize(scs[i].cycle)
            _bars(gs[i], os_[i], rs[i], ro, len(scs[i].critics), label)
            u = _fp64(label, cfgs[i], css[i], nzs[i], gs[i].get_costs(), _controls(rs[i]))
            assert u.saturated() == _want_saturated(cfgs[i]), f"{label}: {u.saturated()}"
            _check_coupling(cfgs[i], [u], label)
    for e in gs + os_:
        e.close()


# ------------------------------------------------------------------------------------------------
# B. speed limits changed between cycles
# ------------------------------------------------------------------------------------------------
LIMITS = [None, (0.21, False), (37.0, True), (0.0, False)]   # per cycle: none, absolute, percentage, NO_SPEED_LIMIT


@pytest.mark.parametrize("path", ["fused", "stream_tma", "stream_b4r3", "group", "group_device"])
@pytest.mark.parametrize("profile", ["omni", "ackermann_r0.75"])
def test_speed_limit(product_fns, oracle_fns, monkeypatch, profile, path):
    """the clip follows the speed-limited constraints; ConstraintCritic keeps the base ones (its rows against the
    oracle's, constraint_critic.cpp:31-38).  In a group the member records rebuild after every change."""
    B, env = (1000, {}) if path.startswith("group") or path == "fused" else (PATHS[path][0], STREAM)
    cfgs = [ps.profile_cfg(profile, B, T)] + ([ps.profile_cfg("omni_vxmin_pos", 700, T)] if path.startswith("group") else [])
    scs = [ps.scene(c, seed=60 + i) for i, c in enumerate(cfgs)]
    nzs = [ps.noise(c, 60 + i) for i, c in enumerate(cfgs)]
    gs = [_engine(product_fns, sc, nz, env, monkeypatch) for sc, nz in zip(scs, nzs)]
    os_ = [_engine(oracle_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    if path == "group_device":
        for e in gs:
            e.set_costmap_residency(True)
    hs = _bind(product_fns, gs) if path.startswith("group") else None
    constraint_q = [q for q, (n, _) in enumerate(scs[0].critics) if n == "ConstraintCritic"]
    assert constraint_q
    for cycle, lim in enumerate(LIMITS):
        if lim is not None:
            for e in gs + os_:
                e.set_speed_limit(*lim)
        lims = [ps.limits(c, *lim) if lim else ps.limits(c) for c in cfgs]
        css = [ps.warm_start(c, l) for c, l in zip(cfgs, lims)]
        for e, f, cs in zip(gs, os_, css):
            e.set_control_sequence(*cs)
            f.set_control_sequence(*cs)
        if path == "group":
            rs = _host_batch(product_fns, gs, hs, [sc.cycle for sc in scs])
        elif path == "group_device":
            rs = optimize_group_device(gs, *_inputs([_on_device(sc.cycle) for sc in scs]))
        else:
            rs = [gs[0].optimize(scs[0].cycle)]
        for i in range(len(gs)):
            label = f"{profile} {path} member {i} cycle {cycle} limit {lim}"
            got = gs[i].get_constraints()
            np.testing.assert_allclose([got[k] for k in ("vx_max", "vx_min", "vy", "wz")], lims[i], rtol=1e-6, err_msg=label)
            ro = os_[i].optimize(scs[i].cycle)
            _bars(gs[i], os_[i], rs[i], ro, len(scs[i].critics), label)
            u = _fp64(label, cfgs[i], css[i], nzs[i], gs[i].get_costs(), _controls(rs[i]), lims[i])
            assert u.saturated() == _want_saturated(cfgs[i]), f"{label}: {u.saturated()}"
            assert np.max(np.abs(rs[i].vx)) <= max(abs(lims[i][0]), abs(lims[i][1])) + 1e-6, label
            assert os_[i].get_critic_costs(constraint_q[0]).max() > 0, f"{label}: ConstraintCritic silent"
    for e in gs + os_:
        e.close()


# ------------------------------------------------------------------------------------------------
# C. the critic matrix
# ------------------------------------------------------------------------------------------------
SETTINGS = ps.critic_settings(T)
GATED = ("GoalCritic", "GoalAngleCritic", "PathAlignCritic", "PathAlignLegacyCritic", "PathFollowCritic",
         "PathAngleCritic", "PreferForwardCritic")
MATRIX_PATHS = {"fused": (1000, {}), "two_kernel": (1000, {"MPPI_FUSED": "0"}), "stream": (1000, STREAM),
                "stream_b4r1": (1001, STREAM)}


def _gate_states(o, critics):
    return {n: bool((o.get_critic_costs(q) != 0).any()) for q, (n, d) in enumerate(critics)}


@pytest.mark.parametrize("path", list(MATRIX_PATHS))
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_critic_matrix(product_fns, oracle_fns, monkeypatch, setting, path):
    B, env = MATRIX_PATHS[path]
    cfg = ps.profile_cfg("omni", B, T)
    critics = SETTINGS[setting]
    sc = ps.scene(cfg, critics, seed=21)
    nz = ps.noise(cfg, 21)
    g = _engine(product_fns, sc, nz, env, monkeypatch)
    o = _engine(oracle_fns, sc, nz)
    states = {}
    for cycle in range(2):
        label = f"{setting} {path} cycle {cycle}"
        rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
        _bars(g, o, rg, ro, len(critics), label, control_atol=_control_floor(o, cfg))
        for k, v in _gate_states(o, critics).items():
            states[k] = states.get(k, False) or v
        g.set_control_sequence(*o.get_control_sequence())
    print(f"{setting} {path}: critics with a non-zero row {sorted(k for k, v in states.items() if v)}")
    for n, d in critics:
        if not d.get("enabled", 1):
            assert not states[n], f"{setting}: disabled {n} scored"
    align = states["PathAlignCritic"] and states["PathAlignLegacyCritic"]
    if setting == "power2_gates_closed":
        assert not any(states[n] for n in GATED), states
    elif setting in ("power2", "power3"):
        assert all(states.values()), states
    elif setting.startswith("align_step") and int(setting[10:].split("_")[0]) < T:
        assert align, states
    elif setting.startswith(f"align_step{T + 3}"):
        assert not states["PathAlignCritic"] and not states["PathAlignLegacyCritic"], states   # no sample, disabled
    elif setting.startswith("angle"):
        assert states["PathAngleCritic"] == (not setting.startswith("angle3.12")), states
    elif setting == "occupancy1":
        assert align, states
    g.close(); o.close()


def test_group_of_critic_settings(product_fns, oracle_fns):
    """a bound group whose members run different critic settings (the generic batch instance), host and device inputs"""
    names = ["power2", "power3", "align_step3_yaw1", "align_step56_yaw0", "angle0.0005_fwd0", "angle3.12_fwd1",
             "disabled_middle", "permuted", "deadband2", "offset500"]
    cfg = ps.profile_cfg("omni", 512, T)
    scs = [ps.scene(cfg, SETTINGS[n], seed=80 + i) for i, n in enumerate(names)]
    nzs = [ps.noise(cfg, 80 + i) for i in range(len(names))]
    host = [_engine(product_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    dev = [_engine(product_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    for e in dev:
        e.set_costmap_residency(True)
    os_ = [_engine(oracle_fns, sc, nz) for sc, nz in zip(scs, nzs)]
    hh, _ = _bind(product_fns, host), _bind(product_fns, dev)
    for cycle in range(2):
        rh = _host_batch(product_fns, host, hh, [sc.cycle for sc in scs])
        rd = optimize_group_device(dev, *_inputs([_on_device(sc.cycle) for sc in scs]))
        for i, n in enumerate(names):
            ro = os_[i].optimize(scs[i].cycle)
            for e, r, kind in ((host[i], rh[i], "batch"), (dev[i], rd[i], "device inputs")):
                _bars(e, os_[i], r, ro, len(scs[i].critics), f"{n} {kind} cycle {cycle}", control_atol=_control_floor(os_[i], cfg))
                e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    for e in host + dev + os_:
        e.close()


# ------------------------------------------------------------------------------------------------
# D. softmax extremes
# ------------------------------------------------------------------------------------------------
def _move_argmin(nz, totals, dst, dup=None):
    """swap the rows of the lowest-cost trajectory and row `dst`; dup: also copy it into row `dup` (an exact tie)"""
    b = int(np.argmin(totals))
    out = []
    for a in nz:
        if a is None:
            out.append(None)
            continue
        a = a.copy()
        a[[b, dst]] = a[[dst, b]]
        if dup is not None:
            a[dup] = a[dst]
        out.append(a)
    return out


EXTREMES = {
    # name: (batch, environment, sharded, argmin row, duplicate row)
    "fused_last_tile": (1000, {}, False, 999, None),
    "two_kernel_last_block": (2049, {"MPPI_FUSED": "0"}, False, 2048, None),
    "stream_last_chunk": (4099, STREAM, False, 4098, None),
    "stream_tma_last_chunk": (4096, STREAM, False, 4095, None),
    "second_shard": (1000, {}, True, 998, None),
    "fused_tie_across_tiles": (1000, {}, False, 999, 3),
    "stream_tie_across_chunks": (4099, STREAM, False, 4098, 5),
}


@pytest.mark.parametrize("profile", ["omni_t1e-3", "ackermann_r0.2"])
@pytest.mark.parametrize("case", list(EXTREMES))
def test_low_temperature_argmin_placement(product_fns, oracle_fns, monkeypatch, case, profile):
    """temperature 1e-3: nearly every weight underflows and the minimum sits in the last tile, block, chunk or shard
    (or is tied exactly with a row in the first one)"""
    B, env, sharded, dst, dup = EXTREMES[case]
    cfg = ps.profile_cfg(profile, B, T, temperature=1e-3)
    sc = ps.scene(cfg, seed=31)
    nz0 = ps.noise(cfg, 31)
    probe = _engine(oracle_fns, sc, nz0, outputs=False)
    probe.optimize(sc.cycle)
    nz = _move_argmin(nz0, probe.get_costs(), dst, dup)
    probe.close()
    o = _engine(oracle_fns, sc, nz)
    g = _shards(product_fns, sc, nz) if sharded else _engine(product_fns, sc, nz, env, monkeypatch)
    cs = np.zeros((3, T), np.float32)
    for cycle in range(2):
        label = f"{case} {profile} cycle {cycle}"
        for e in (g if sharded else [g]) + [o]:
            e.set_control_sequence(*cs)
        ro = o.optimize(sc.cycle)
        if sharded:
            rg = optimize_sharded(g, sc.cycle)
            totals = np.concatenate([e.get_costs() for e in g])
            np.testing.assert_allclose(_controls(rg), _controls(ro), rtol=RTOL, atol=ATOL, err_msg=label)
            np.testing.assert_allclose(totals, o.get_costs(), rtol=RTOL, atol=COST_ATOL, err_msg=label)
        else:
            rg = g.optimize(sc.cycle)
            totals = g.get_costs()
            _bars(g, o, rg, ro, len(sc.critics), label)
        u = _fp64(label, cfg, cs, nz, totals, _controls(rg))
        arg = int(np.argmin(totals))
        print(f"{label}: argmin row {arg}, ESS {u.ess:.3f}, weight of the argmin {u.weights[arg]:.4f}")
        assert cycle > 0 or arg in (dst, dup), f"{label}: argmin at {arg}"
        if cycle == 0:
            assert u.ess < 3.0, u.ess
            if dup is not None:
                assert totals[dst] == totals[dup] and abs(u.weights[dst] - u.weights[dup]) < 1e-12
        cs = _controls(ro)
    for e in (g if sharded else [g]) + [o]:
        e.close()


def test_collision_costs_mixed_with_free(product_fns, oracle_fns, monkeypatch):
    """a robot 0.75 m from a ring of discs: 1e6 collision costs next to free trajectories, at temperatures 0.02 and 5,
    fused and stream"""
    for profile in ("omni_t0.02", "omni_t5"):
        for env in ({}, STREAM):
            cfg = ps.profile_cfg(profile, 1000, T)
            critics = ps.critic_list(1, names=("ConstraintCritic", "CostCritic", "PathFollowCritic"),
                                     CostCritic=dict(collision_cost=1.0e6))
            sc = ps.scene(cfg, critics, seed=7, yaw_off=0.0)
            nz = ps.noise(cfg, 7)
            g, o = _engine(product_fns, sc, nz, env, monkeypatch), _engine(oracle_fns, sc, nz)
            label = f"{profile} {env}"
            cs = np.zeros((3, T), np.float32)
            cs[0] = 0.2   # about half of the trajectories reach the discs across the path
            for e in (g, o):
                e.set_control_sequence(*cs)
            rg, ro = g.optimize(sc.cycle), o.optimize(sc.cycle)
            _bars(g, o, rg, ro, len(critics), label)
            totals = g.get_costs()
            _fp64(label, cfg, cs, nz, totals, _controls(rg))
            n_coll = int((totals > 50.0 * totals.min()).sum())
            print(f"{label}: {n_coll} of 1000 trajectories in collision (cost > 50 x the minimum), min total {totals.min():.3f}")
            assert 0 < n_coll < 1000, n_coll
            g.close(); o.close()


# ------------------------------------------------------------------------------------------------
# E. noise with three different stds
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["tile", "stream", "shard_offset"])
@pytest.mark.parametrize("profile", ["omni", "diff", "ackermann_r0.2"])
def test_philox_noise_three_stds(product_fns, oracle_fns, monkeypatch, profile, layout):
    kw = dict(seed=4321)
    if layout == "shard_offset":
        kw.update(shard_offset=333, shard_total=5000)
    cfg = ps.profile_cfg(profile, 1000, T, **kw)
    env = STREAM if layout == "stream" else {}
    _set_env(monkeypatch, env)
    g = Engine(product_fns, **cfg)
    _clear_env(monkeypatch, env)
    o = Engine(oracle_fns, **cfg)
    g.generate_noise(3)
    o.generate_noise(3)
    stds = (cfg["vx_std"], cfg["vy_std"], cfg["wz_std"])
    for p, (a, b, s) in enumerate(zip(g.get_noise(), o.get_noise(), stds)):
        if p == 1 and not ps.holonomic(cfg):
            assert not a.any(), "the lateral plane of a non-holonomic model is not zero"
            continue
        np.testing.assert_allclose(a, b, rtol=0, atol=2e-6 * s / 0.2, err_msg=f"plane {p}")
        assert abs(float(a.std()) - s) < 0.02 * s, (p, float(a.std()), s)
    g.close(); o.close()


def test_group_regenerate_noises_three_stds(product_fns, oracle_fns):
    """regenerate_noises members of a bound group redraw with their own three stds (the group's redraw table)"""
    cfgs = [ps.profile_cfg(n, 512, T, iteration_count=2, regenerate_noises=1, seed=9 + i)
            for i, n in enumerate(("omni", "omni_gamma0.3", "diff"))]
    scs = [ps.scene(c, seed=90 + i) for i, c in enumerate(cfgs)]
    gs, os_ = [], []
    for sc in scs:
        for fns, lst in ((product_fns, gs), (oracle_fns, os_)):
            e = Engine(fns, **sc.cfg)
            e.set_robot(sc.robot)
            e.set_critics(sc.critics)
            e.generate_noise(0)
            lst.append(e)
    hs = _bind(product_fns, gs)
    _host_batch(product_fns, gs, hs, [sc.cycle for sc in scs])
    for sc, o in zip(scs, os_):
        o.optimize(sc.cycle)
    for i, (g, o) in enumerate(zip(gs, os_)):
        stds = (cfgs[i]["vx_std"], cfgs[i]["vy_std"], cfgs[i]["wz_std"])
        for p, (a, b, s) in enumerate(zip(g.get_noise(), o.get_noise(), stds)):
            np.testing.assert_allclose(a, b, rtol=0, atol=2e-6 * s / 0.2, err_msg=f"member {i} plane {p}")
            if p == 1 and not ps.holonomic(cfgs[i]):
                assert not a.any()
            else:
                assert abs(float(a.std()) - s) < 0.03 * s, (i, p, float(a.std()), s)
    for e in gs + os_:
        e.close()


# ------------------------------------------------------------------------------------------------
# F. batches beyond 65535 row blocks of 32: the noise transposes and merges of more partial records than
#    merge_finalize_body caches
# ------------------------------------------------------------------------------------------------
BIG_B, BIG_T = 2_100_001, 8   # (B + 31) / 32 = 65626 row blocks; B / 1024 + 1 = 2051 chunk records (kMergeCached = 2048)


def test_noise_transposes_of_a_big_batch(product_fns, monkeypatch):
    """mppi_set_noise into the stream layout and to_stream_layout (mppi_batch_bind of a tile-layout handle) transpose
    [B][T] -> [T][B]; mppi_get_noise transposes back.  Both directions, bit for bit, at a batch size whose row blocks do
    not fit in one grid's y dimension."""
    rng = np.random.default_rng(71)
    nz = [rng.standard_normal((BIG_B, BIG_T)).astype(np.float32) for _ in range(3)]
    cfg = ps.profile_cfg("omni", BIG_B, BIG_T)
    for layout, env in (("stream", STREAM), ("tile, then bound", {"MPPI_STREAM_MIN_BATCH": str(4 * BIG_B)})):
        _set_env(monkeypatch, env)
        e = Engine(product_fns, **cfg)
        _clear_env(monkeypatch, env)
        e.set_noise(*nz)
        if layout != "stream":
            _bind(product_fns, [e])
        for p, (a, b) in enumerate(zip(e.get_noise(), nz)):
            bad = np.flatnonzero(a != b)
            assert bad.size == 0, f"{layout}: plane {p}: {bad.size} values differ, first row {bad[0] // BIG_T}"
        e.close()


def _move_lowest(nz, totals, dst):
    """the noise rows permuted so that the len(dst) lowest-cost trajectories sit in rows dst (costs are per row: the
    permutation moves them with their rows)"""
    B = totals.shape[0]
    low = np.argsort(totals, kind="stable")[:len(dst)]
    order = np.empty(B, np.int64)
    mask = np.zeros(B, bool)
    mask[dst] = True
    order[dst] = low
    order[~mask] = np.setdiff1d(np.arange(B), low)
    return [None if a is None else a[order] for a in nz]


# layout: (batch, time steps, environment, first row of the uncached records).  The stream layout's chunk records all
# carry the global minimum (K3 publishes it first), so there every rescale factor is 1 and the uncached branch only
# re-derives it; in the tile layout every K3 block of kUpdRows = 32 rows records its own minimum, and a wrong factor
# for a record beyond the cache shows.
MERGE_LAYOUTS = {
    "stream": (BIG_B, BIG_T, STREAM, 2048 * 1024),
    "tile_two_kernel": (2050 * 32 - 27, BIG_T, {"MPPI_FUSED": "0", "MPPI_STREAM_MIN_BATCH": str(10 ** 8)}, 2048 * 32),
}


@pytest.mark.parametrize("layout", list(MERGE_LAYOUTS))
@pytest.mark.parametrize("profile", ["omni", "ackermann_r0.75"])
def test_merge_beyond_cached_records(product_fns, oracle_fns, monkeypatch, profile, layout):
    """merge_finalize_kernel over more partial records than the kMergeCached = 2048 rescale factors it caches: the
    stream layout at T = 8, B = 2 100 001 (B % 4 != 0: 2051 chunk records of 1024 trajectories) and the two-kernel tile
    layout at B = 65 573 (2050 K3 blocks of 32).  Temperature 1e-3 with the lowest-cost trajectories moved into the
    records beyond the cache, warm start beyond every bound.  The oracle accumulates in double (set_wide_reductions);
    the rule of test_config4_full_size_against_the_oracle applies to the controls: closer to the order-free value than
    the index-order float oracle, or within 1e-5 of it."""
    B, Tl, env, uncached = MERGE_LAYOUTS[layout]
    cfg = ps.profile_cfg(profile, B, Tl, temperature=1e-3)
    critics = ps.critic_list(2, names=("ConstraintCritic", "CostCritic", "GoalCritic", "PathFollowCritic"),
                             CostCritic=dict(consider_footprint=0))
    sc = ps.scene(cfg, critics, seed=51)
    nz0 = ps.noise(cfg, 51)
    cs = ps.warm_start(cfg, period=1)
    g = _engine(product_fns, sc, nz0, env, monkeypatch, outputs=False)
    g.set_control_sequence(*cs)
    g.optimize(sc.cycle)
    n_low = min(64, B - uncached)
    nz = _move_lowest(nz0, g.get_costs(), np.arange(B - n_low, B))
    g.set_noise(*nz)
    o = _engine(oracle_fns, sc, nz, outputs=False)
    oracle_fns["set_wide_reductions"](o.h, 1)
    lit = _engine(oracle_fns, sc, nz, outputs=False)
    for e in (g, o, lit):
        e.set_control_sequence(*cs)
    rg, ro, rl = g.optimize(sc.cycle), o.optimize(sc.cycle), lit.optimize(sc.cycle)
    totals = g.get_costs()
    np.testing.assert_allclose(totals, o.get_costs(), rtol=RTOL, atol=COST_ATOL)
    d_dev = float(np.abs(_controls(rg) - _controls(ro)).max())
    d_lit = float(np.abs(_controls(rl) - _controls(ro)).max())
    u = ps.update_fp64(cs, ps.noise_planes(nz, cfg), totals, dict(cfg, gamma=0.0))
    d_fp64 = float(np.abs(_controls(rg) - u.controls).max())
    w_tail = float(u.weights[uncached:].sum())
    print(f"{profile} {layout}: argmin row {int(np.argmin(totals))}, ESS {u.ess:.2f}, weight of the uncached records "
          f"{w_tail:.3f}, device vs order-free {d_dev:.2e}, index-order vs order-free {d_lit:.2e}, device vs update_fp64 "
          f"{d_fp64:.2e}, saturated {sorted(u.saturated())}, coupled steps {int(u.coupled.sum())}")
    assert int(np.argmin(totals)) >= uncached
    assert w_tail > 0.5, "the uncached records carry too little weight to show a wrong rescale factor"
    assert d_dev < d_lit or d_dev < 1e-5, (d_dev, d_lit)
    assert d_fp64 < 1e-5, d_fp64
    assert u.saturated() == _want_saturated(cfg)
    _check_coupling(cfg, [u], profile)
    for e in (g, o, lit):
        e.close()

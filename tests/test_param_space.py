"""CPU checks of tests/param_space.py: the oracle's update equals update_fp64 on every profile, the profiles are
asymmetric, and the saturating scenes reach every bound they claim (counted by update_fp64 on the oracle's own costs)."""
import itertools

import numpy as np
import pytest

from mpcholonavigation_b200 import Engine
from tests import param_space as ps

B, T = 256, 24


def _oracle_cycle(oracle_fns, cfg, critics=None, seed=3, lims=None):
    sc = ps.scene(cfg, critics, seed)
    nz = ps.noise(cfg, seed)
    o = Engine(oracle_fns, **cfg)
    o.set_robot(sc.robot)
    o.set_critics(sc.critics)
    o.set_noise(*nz)
    o.set_outputs(critic_costs=True)
    cs = ps.warm_start(cfg, lims)
    o.set_control_sequence(*cs)
    r = o.optimize(sc.cycle)
    rows = sum(o.get_critic_costs(q).astype(np.float64) for q in range(len(sc.critics)))
    out = (cs, ps.noise_planes(nz, cfg), o.get_costs(), rows, np.stack([r.vx, r.vy, r.wz]))
    o.close()
    return out


@pytest.mark.parametrize("profile", list(ps.PROFILES))
def test_oracle_update_equals_update_fp64(oracle_fns, profile):
    cfg = ps.profile_cfg(profile, B, T)
    cs, nz, total, rows, got = _oracle_cycle(oracle_fns, cfg)
    # the softmax, weighted sums and clip alone: the oracle's totals (gamma included) through the fp64 update
    u = ps.update_fp64(cs, nz, total, dict(cfg, gamma=0.0))
    np.testing.assert_allclose(got, u.controls, rtol=1e-5, atol=2e-6)
    # the gamma term with the profile's three stds
    np.testing.assert_allclose(total - rows, ps.gamma_term_fp64(cs, nz, cfg), rtol=1e-4, atol=2e-4 * max(1.0, np.abs(total).max() * 1e-3))
    if not ps.holonomic(cfg):
        assert np.array_equal(got[1], cs[1])


def test_profiles_are_asymmetric():
    cfgs = {n: ps.profile_cfg(n, B, T) for n in ps.PROFILES}
    for n, cfg in cfgs.items():
        assert all(ps.asymmetry(cfg).values()), (n, ps.asymmetry(cfg))
    for a, b in itertools.combinations(cfgs, 2):
        assert cfgs[a] != cfgs[b], (a, b)
    vx_min = {cfg["vx_min"] for cfg in cfgs.values()}
    assert min(vx_min) < 0 and 0.0 in vx_min and max(vx_min) > 0
    temps = {cfg["temperature"] for cfg in cfgs.values()}
    assert {1e-3, 0.02, 5.0} <= temps and {0.0, 0.3} <= {cfg["gamma"] for cfg in cfgs.values()}
    assert {cfg["motion_model"] for cfg in cfgs.values()} == {"Omni", "Ackermann", "DiffDrive"}
    assert {cfg["ackermann_min_turning_r"] for cfg in cfgs.values() if cfg["motion_model"] == "Ackermann"} == {0.2, 0.75}


@pytest.mark.parametrize("profile", list(ps.PROFILES))
def test_warm_start_saturates_every_bound(oracle_fns, profile):
    """each plane's high and low bound clips somewhere in the horizon; the Ackermann coupling acts"""
    cfg = ps.profile_cfg(profile, B, T)
    cs, nz, total, rows, got = _oracle_cycle(oracle_fns, cfg)
    u = ps.update_fp64(cs, nz, total, dict(cfg, gamma=0.0))
    planes = (0, 1, 2) if ps.holonomic(cfg) else (0, 2)
    assert u.saturated() == {(p, s) for p in planes for s in (-1, 1)}, u.saturated()
    if cfg["motion_model"] == "Ackermann":
        assert u.coupled.sum() >= 4
        if cfg["ackermann_min_turning_r"] > 0.5:   # coupled where vx sits on its bound, too
            assert (u.coupled & (u.hits[0] != 0)).any()
    else:
        assert not u.coupled.any()


@pytest.mark.parametrize("speed_limit,percentage", [(0.21, False), (37.0, True)])
def test_warm_start_saturates_speed_limited_bounds(oracle_fns, speed_limit, percentage):
    cfg = ps.profile_cfg("omni", B, T)
    lims = ps.limits(cfg, speed_limit, percentage)
    sc = ps.scene(cfg)
    o = Engine(oracle_fns, **cfg)
    o.set_robot(sc.robot)
    o.set_critics(sc.critics)
    nz = ps.noise(cfg, 5)
    o.set_noise(*nz)
    o.set_speed_limit(speed_limit, percentage)
    got_lims = o.get_constraints()
    np.testing.assert_allclose([got_lims[k] for k in ("vx_max", "vx_min", "vy", "wz")], lims, rtol=1e-6)
    cs = ps.warm_start(cfg, lims)
    o.set_control_sequence(*cs)
    r = o.optimize(sc.cycle)
    u = ps.update_fp64(cs, ps.noise_planes(nz, cfg), o.get_costs(), dict(cfg, gamma=0.0), lims)
    np.testing.assert_allclose(np.stack([r.vx, r.vy, r.wz]), u.controls, rtol=1e-5, atol=2e-6)
    assert len(u.saturated()) == 6
    assert np.abs(u.controls[0]).max() <= max(abs(lims[0]), abs(lims[1])) + 1e-7
    o.close()


def test_critic_settings_are_accepted_by_the_oracle(oracle_fns):
    """every critic list of critic_settings configures and runs to finite costs (PathAlign steps up to T + 3 included)"""
    cfg = ps.profile_cfg("omni", 64, T)
    for name, critics in ps.critic_settings(T).items():
        _, _, total, rows, _ = _oracle_cycle(oracle_fns, cfg, critics)
        assert np.isfinite(total).all(), name

"""Optimizer profiles and critic settings away from the deployed values, the float64 update they are checked against,
and scenes whose warm start drives the update past every bound.  TEST INFRASTRUCTURE: nothing under
mpcholonavigation_b200/ imports this.

The deployed optimizer setting (scenarios._omni_cfg) has vx_std == vy_std and vx_max == vy_max, so a kernel that reads
the wrong field of either pair computes the same numbers.  Every profile below has three distinct stds, three distinct
limits and a non-round dt, so that any swap of two fields changes the result.

update_fp64 is tests/golden/make_vectors.py's softmax_update with the Ackermann coupling of
motion_models.hpp:110-117 behind the clip, and it reports which bound each (plane, t) hit and where the coupling acted.
"""
import dataclasses

import numpy as np

from mpcholonavigation_b200 import scenarios

# ------------------------------------------------------------------------------------------------
# optimizer profiles
# ------------------------------------------------------------------------------------------------
_BASE = dict(model_dt=0.043, iteration_count=1, temperature=0.27, gamma=0.021, vx_max=0.55, vx_min=-0.31, vy_max=0.37,
             wz_max=1.63, vx_std=0.23, vy_std=0.17, wz_std=0.41, motion_model="Omni", ackermann_min_turning_r=0.2)

PROFILES = {
    "omni": {},
    "omni_vxmin_zero": dict(vx_min=0.0),
    "omni_vxmin_pos": dict(vx_min=0.07),
    "omni_t1e-3": dict(temperature=1e-3),
    "omni_t0.02": dict(temperature=0.02),
    "omni_t5": dict(temperature=5.0),
    "omni_gamma0": dict(gamma=0.0),
    "omni_gamma0.3": dict(gamma=0.3),
    "ackermann_r0.2": dict(motion_model="Ackermann", ackermann_min_turning_r=0.2),
    "ackermann_r0.75": dict(motion_model="Ackermann", ackermann_min_turning_r=0.75),
    "diff": dict(motion_model="DiffDrive"),
}


def profile_cfg(name, batch, steps, **kw):
    return {**_BASE, **PROFILES[name], "batch_size": batch, "time_steps": steps, **kw}


def holonomic(cfg):
    return cfg["motion_model"] == "Omni"


def limits(cfg, speed_limit=None, percentage=False):
    """(vx_max, vx_min, vy, wz) that the clip uses: mppi_set_speed_limit (ratio of the base limits) or the base ones"""
    base = np.array([cfg["vx_max"], cfg["vx_min"], cfg["vy_max"], cfg["wz_max"]], np.float32)
    if not speed_limit:
        return tuple(float(v) for v in base)
    ratio = speed_limit / 100.0 if percentage else speed_limit / float(base[0])
    return tuple(float(np.float32(float(v) * ratio)) for v in base)


def asymmetry(cfg):
    """the pairs that must differ so that a swap of two fields shows"""
    stds = (cfg["vx_std"], cfg["vy_std"], cfg["wz_std"])
    lims = (cfg["vx_max"], cfg["vy_max"], cfg["wz_max"], abs(cfg["vx_min"]))
    return dict(stds_distinct=len(set(stds)) == 3, limits_distinct=len(set(lims)) == 4,
                dt_not_round=round(cfg["model_dt"], 2) != cfg["model_dt"])


# ------------------------------------------------------------------------------------------------
# the update in float64
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Update:
    controls: np.ndarray    # [3][T]
    costs: np.ndarray       # [B] with the gamma term
    weights: np.ndarray     # [B], normalised
    hits: np.ndarray        # [3][T] int8: -1 the low bound clipped, +1 the high bound, 0 inside
    coupled: np.ndarray     # [T] bool: the Ackermann coupling replaced wz

    @property
    def ess(self):
        """effective sample size of the softmax weights"""
        return float(1.0 / np.sum(self.weights ** 2))

    def saturated(self):
        """{(plane, side)} hit anywhere in the horizon; plane 0 vx, 1 vy, 2 wz; side -1 low, +1 high"""
        return {(p, int(s)) for p in range(3) for s in (-1, 1) if (self.hits[p] == s).any()}


def update_fp64(cs, noise, costs, cfg, lims=None):
    """Optimizer::updateControlSequence + applyControlSequenceConstraints (optimizer.cpp:362-394, 237-249) and
    AckermannMotionModel::applyConstraints (motion_models.hpp:110-117), float64.
    cs [3][T] (vx, vy, wz), noise [3][B][T], costs [B] (critic costs before the gamma term; pass the device's totals with
    gamma = 0 in cfg to check the softmax alone).  lims: (vx_max, vx_min, vy, wz), default the profile's base limits."""
    hol = holonomic(cfg)
    cs = np.asarray(cs, np.float64)
    c = cs[:, None, :] + np.asarray(noise, np.float64)
    costs = np.asarray(costs, np.float64).copy()
    std = (cfg["vx_std"], cfg["vy_std"], cfg["wz_std"])
    planes = (0, 2, 1) if hol else (0, 2)
    for p in planes:
        costs += cfg["gamma"] / float(np.float32(std[p])) ** 2 * np.sum(cs[p][None, :] * (c[p] - cs[p][None, :]), axis=1)
    w = np.exp(-(costs - costs.min()) / float(np.float32(cfg["temperature"])))
    w /= w.sum()
    new = cs.copy()
    for p in planes:
        new[p] = (w[:, None] * c[p]).sum(axis=0)
    vx_max, vx_min, vy, wz = lims if lims is not None else limits(cfg)
    lo = np.array([vx_min, -vy, -wz])
    hi = np.array([vx_max, vy, wz])
    hits = np.zeros((3, cs.shape[1]), np.int8)
    for p in planes:
        hits[p] = np.where(new[p] < lo[p], -1, np.where(new[p] > hi[p], 1, 0))
        new[p] = np.clip(new[p], lo[p], hi[p])
    coupled = np.zeros(cs.shape[1], bool)
    if cfg["motion_model"] == "Ackermann":
        r = float(np.float32(cfg["ackermann_min_turning_r"]))
        with np.errstate(divide="ignore", invalid="ignore"):
            coupled = np.abs(new[0]) / np.abs(new[2]) < r
        new[2] = np.where(coupled, np.sign(new[2]) * np.abs(new[0]) / r, new[2])
    return Update(new, costs, w, hits, coupled)


def gamma_term_fp64(cs, noise, cfg):
    """the gamma term of every trajectory alone (what the total cost holds beyond the critic rows)"""
    out = np.zeros(np.asarray(noise).shape[1])
    std = (cfg["vx_std"], cfg["vy_std"], cfg["wz_std"])
    for p in ((0, 2, 1) if holonomic(cfg) else (0, 2)):
        k = float(np.float32(np.float32(cfg["gamma"]) / np.float32(std[p]) ** 2))
        out += k * np.sum(np.asarray(cs[p], np.float64)[None, :] * np.asarray(noise[p], np.float64), axis=1)
    return out


# ------------------------------------------------------------------------------------------------
# scenes
# ------------------------------------------------------------------------------------------------
def warm_start(cfg, lims=None, period=4):
    """A control sequence beyond the bounds: plane p at time t is above its high bound, below its low bound or inside,
    in blocks of `period` steps, the pattern shifted by plane so that no two planes hit the same bound at the same t.
    Beyond means by 1.25 x the bound plus three stds, so that the softmax mean of cs + noise stays beyond it at any
    temperature.  Inside is small for vx and 0.6 wz_max for wz, so that the Ackermann coupling acts there."""
    T = cfg["time_steps"]
    vx_max, vx_min, vy, wz = lims if lims is not None else limits(cfg)
    std = (cfg["vx_std"], cfg["vy_std"], cfg["wz_std"])
    lo, hi = (vx_min, -vy, -wz), (vx_max, vy, wz)
    inside = (min(max(0.04, vx_min + 0.01), vx_max - 0.01), 0.3 * vy, 0.6 * wz)
    cs = np.zeros((3, T), np.float32)
    for p in range(3):
        for t in range(T):
            k = (t // period + 2 * p) % 3
            span = 0.25 * (hi[p] - lo[p]) + 3.0 * std[p]
            cs[p, t] = (hi[p] + span, lo[p] - span, inside[p] if (t // period) % 2 == 0 else -inside[p])[k]
    if not holonomic(cfg):
        cs[1] = 0.0
    return cs


def noise(cfg, seed):
    """injected noise with the profile's stds; no lateral plane for a non-holonomic model"""
    B, T = cfg["batch_size"], cfg["time_steps"]
    z = np.random.default_rng(seed).standard_normal((3, B, T)).astype(np.float32)
    vx, vy, wz = (z[i] * np.float32(cfg[k]) for i, k in enumerate(("vx_std", "vy_std", "wz_std")))
    return (vx, vy if holonomic(cfg) else None, wz)


def noise_planes(nz, cfg):
    """the injected noise as [3][B][T] float64 (zeros for the missing lateral plane)"""
    vx, vy, wz = nz
    return np.stack([vx, np.zeros_like(vx) if vy is None else vy, wz]).astype(np.float64)


def scene(cfg, critics=None, seed=1, yaw_off=1.1):
    """config1's map and path with a ring of discs 0.75 m around the robot (two of them across the path), the robot
    turned `yaw_off` rad away from the path (so that PathAngle scores), under the profile `cfg`; critics default to the
    deployed Omni set"""
    sc = scenarios.config1(batch=cfg["batch_size"], steps=cfg["time_steps"], noise_seed=seed, ring=0.75)
    x, y, yaw = sc.cycle.pose
    cyc = dataclasses.replace(sc.cycle, pose=(x, y, yaw + yaw_off))
    return scenarios.Scenario(sc.name, dict(cfg), critics if critics is not None else sc.critics, sc.robot, cyc, seed)


# ------------------------------------------------------------------------------------------------
# critic settings
# ------------------------------------------------------------------------------------------------
ALL_CRITICS = ("ConstraintCritic", "CostCritic", "GoalCritic", "GoalAngleCritic", "ObstaclesCritic", "PathAlignCritic",
               "PathAlignLegacyCritic", "PathFollowCritic", "PathAngleCritic", "PreferForwardCritic", "TwirlingCritic",
               "VelocityDeadbandCritic")
# distinct, non-round weights
WEIGHTS = dict(zip(ALL_CRITICS, (3.7, 2.9, 4.3, 2.3, 1.7, 11.3, 7.9, 4.1, 2.7, 3.3, 6.1, 13.7)))
# thresholds that open every distance gate on config1 (goal 1.95 m from the robot); GATES_CLOSED closes them
OPEN = dict(GoalCritic=dict(threshold_to_consider=2.5), GoalAngleCritic=dict(threshold_to_consider=2.5),
            PathAlignCritic=dict(threshold_to_consider=0.3), PathAlignLegacyCritic=dict(threshold_to_consider=0.3),
            PathFollowCritic=dict(threshold_to_consider=0.3), PathAngleCritic=dict(threshold_to_consider=0.3),
            PreferForwardCritic=dict(threshold_to_consider=0.3))
CLOSED = dict(GoalCritic=dict(threshold_to_consider=0.4), GoalAngleCritic=dict(threshold_to_consider=0.4),
              PathAlignCritic=dict(threshold_to_consider=2.5), PathAlignLegacyCritic=dict(threshold_to_consider=2.5),
              PathFollowCritic=dict(threshold_to_consider=2.5), PathAngleCritic=dict(threshold_to_consider=2.5),
              PreferForwardCritic=dict(threshold_to_consider=2.5))
_COMMON = dict(
    CostCritic=dict(consider_footprint=1, critical_cost=270.0, collision_cost=7.5e5, near_goal_distance=0.7),
    ObstaclesCritic=dict(consider_footprint=1, cost_scaling_factor=3.0, repulsion_weight=1.7, critical_weight=23.0,
                         collision_margin_distance=0.13, near_goal_distance=0.45, collision_cost=9.1e4),
    PathAlignCritic=dict(offset_from_furthest=6, trajectory_point_step=4, max_path_occupancy_ratio=0.3),
    PathAlignLegacyCritic=dict(offset_from_furthest=6, trajectory_point_step=4, max_path_occupancy_ratio=0.3),
    PathFollowCritic=dict(offset_from_furthest=5),
    PathAngleCritic=dict(offset_from_furthest=4, max_angle_to_furthest=1.0),
    VelocityDeadbandCritic=dict(deadband_velocities=[0.07, 0.13, 0.29]),
)


def critic_list(power=1, gates=OPEN, names=ALL_CRITICS, **over):
    """all twelve critics (or `names` in that order) with distinct weights, `power`, the gates of `gates` and per-critic
    overrides over={name: {param: value}}"""
    out = []
    for n in names:
        d = dict(cost_power=power, cost_weight=WEIGHTS[n], **_COMMON.get(n, {}))
        d.update(gates.get(n, {}))
        d.update(over.get(n, {}))
        out.append((n, d))
    return out


def critic_settings(T):
    """name -> critic list, each one a corner of the critics' parameter space"""
    s = {"power1": critic_list(1), "power2": critic_list(2), "power3": critic_list(3),
         "power2_gates_closed": critic_list(2, CLOSED)}
    for step in (1, 2, 3, 5, 7, T):
        for yaw in (0, 1):
            p = dict(trajectory_point_step=step, use_path_orientations=yaw)
            s[f"align_step{step}_yaw{yaw}"] = critic_list(2, PathAlignCritic=p, PathAlignLegacyCritic=p)
    # a step beyond the horizon: PathAlign takes no sample at all.  PathAlignLegacy is disabled there: it divides by
    # floor(T / step) = 0 (path_align_legacy_critic.cpp), so its cost is 0 / 0 = NaN in the reference as in the kernels
    for yaw in (0, 1):
        p = dict(trajectory_point_step=T + 3, use_path_orientations=yaw)
        s[f"align_step{T + 3}_yaw{yaw}"] = critic_list(2, PathAlignCritic=p, PathAlignLegacyCritic=dict(p, enabled=0))
    for ratio in (0.0, 1.0):
        p = dict(max_path_occupancy_ratio=ratio)
        s[f"occupancy{ratio:g}"] = critic_list(2, PathAlignCritic=p, PathAlignLegacyCritic=p)
    for off in (0, 500):
        p = dict(offset_from_furthest=off)
        s[f"offset{off}"] = critic_list(3, PathAlignCritic=p, PathAlignLegacyCritic=p, PathFollowCritic=p,
                                        PathAngleCritic=p)
    for thr in (5e-4, 0.3, 3.12):
        for fwd in (0, 1):
            s[f"angle{thr:g}_fwd{fwd}"] = critic_list(2, PathAngleCritic=dict(max_angle_to_furthest=thr, forward_preference=fwd))
    s["obstacles_point"] = critic_list(2, ObstaclesCritic=dict(consider_footprint=0, repulsion_weight=3.1, critical_weight=7.0,
                                                                collision_margin_distance=0.31, near_goal_distance=3.0))
    s["cost_point"] = critic_list(3, CostCritic=dict(consider_footprint=0, critical_cost=90.0, collision_cost=2.5e3,
                                                      near_goal_distance=3.0))
    for i, db in enumerate(([0.31, 0.02, 0.11], [0.0, 0.29, 0.5], [0.53, 0.41, 1.7])):
        s[f"deadband{i}"] = critic_list(2, VelocityDeadbandCritic=dict(deadband_velocities=db))
    s["disabled_middle"] = critic_list(2, PathAlignCritic=dict(enabled=0), ObstaclesCritic=dict(enabled=0))
    s["permuted"] = critic_list(2, names=ALL_CRITICS[::-1][6:] + ALL_CRITICS[::-1][:6])
    return s

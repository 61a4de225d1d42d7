"""Bound robot groups (mppi_batch_bind) whose members run with iteration_count > 1 or regenerate_noises: the group's
batched launches serve them, with the same results as the one-by-one path.

- iteration_count = 2: each member against its own CPU oracle (the bars of test_iteration_count_two: the second
  rollout starts from an update whose reduction order differs from the oracle's).
- regenerate_noises: each member against an unbound twin (same configuration and seed, mppi_optimize); after every
  cycle the twin holds bit for bit the noise set the member holds, and that stays so after mppi_batch_unbind.
- A group whose members differ in iteration_count runs them one by one and still matches the oracle.

66 members: two chunks of 64 robots, so that every per-chunk step (redraw between iterations, packet delivery of the
last iteration only) and the single redraw behind the last chunk are exercised.
"""
import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, abi, scenarios

pytestmark = pytest.mark.gpu

RTOL, ATOL, COST_ATOL = 1e-4, 1e-6, 2e-6        # the bars of the iteration_count = 1 group test
RTOL2, ATOL2 = 1e-3, 1e-5                       # iteration_count = 2 (test_iteration_count_two)
N_MEMBERS = 66
CHUNKS = 2                                      # of 64 robots


def _engine(fns, sc, noise=None, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise is not None:
        e.set_noise(*noise)
    return e


def _bind(fns, engines):
    hs = (abi.H * len(engines))(*[e.h for e in engines])
    assert fns["batch_bind"](hs, len(engines)) == 0
    return hs


def _group_io(scs):
    n, T = len(scs), scs[0].cfg["time_steps"]
    ins, outs = (abi.CycleIn * n)(), (abi.CycleOut * n)()
    keep, bufs = [], []
    for i, sc in enumerate(scs):
        cin, k = sc.cycle.pack()
        ins[i] = cin
        arrs = [np.empty(T, np.float32) for _ in range(3)]
        outs[i].control_vx, outs[i].control_vy, outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
        keep.append(k); bufs.append(arrs)
    return ins, outs, keep, bufs


def _launches(engines):
    return sum(e.get_profile()["kernel_launches"] for e in engines)


def _check_against_oracle(label, bufs, out, g, o, ro, iterations):
    rtol, atol = (RTOL, ATOL) if iterations == 1 else (RTOL2, ATOL2)
    for a, name in zip(bufs, ("vx", "vy", "wz")):
        np.testing.assert_allclose(a, getattr(ro, name), rtol=rtol, atol=atol, err_msg=f"{label} {name}")
    assert bool(out.fail_flag) == bool(ro.fail_flag), label
    want = abi.UINT32_MAX if ro.furthest_reached_path_point is None else ro.furthest_reached_path_point
    assert out.furthest_reached_path_point == want, label
    cg, co = g.get_costs(), o.get_costs()
    if iterations == 1:
        np.testing.assert_allclose(cg, co, rtol=RTOL, atol=COST_ATOL, err_msg=f"{label} costs")
    else:
        # the second rollout may move a trajectory onto another cell: a handful of totals differ (2 of 256 allowed there)
        bad = ~np.isclose(cg, co, rtol=1e-3, atol=1e-4)
        assert bad.sum() <= max(2, cg.size // 100), (label, int(bad.sum()))


def test_iteration_count_two_group_against_the_oracle(product_fns, oracle_fns):
    """iteration_count = 2 in a bound group of 66 robots, 4 cycles: every member's controls, fail flag, furthest point
    and accumulated costs (quirk R20) against its own oracle; the batched launches ran (4 per iteration per chunk)."""
    scs = [scenarios.config5_robot(r) for r in range(N_MEMBERS)]
    for sc in scs:
        sc.cfg["iteration_count"] = 2
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    orcs = [_engine(oracle_fns, sc, sc.noise()) for sc in scs]
    hs = _bind(product_fns, group)
    ins, outs, keep, bufs = _group_io(scs)
    launches0 = _launches(group)
    for cycle in range(4):
        assert product_fns["optimize_batch"](hs, ins, outs, N_MEMBERS) == 0
        for i, (sc, o) in enumerate(zip(scs, orcs)):
            ro = o.optimize(sc.cycle)
            _check_against_oracle(f"cycle {cycle} robot {i}", bufs[i], outs[i], group[i], o, ro, 2)
            group[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    # 4 cycles x 2 chunks x 2 iterations x 4 launches; one by one it would be 66 robots x 2 iterations x 3 per cycle
    assert _launches(group) - launches0 == 4 * CHUNKS * 2 * 4
    for e in group + orcs:
        e.close()


def _regen_group(fns, iterations, regen):
    """a bound group and, for every member that regenerates its noise, an unbound twin with the same seed"""
    scs = [scenarios.config5_robot(r) for r in range(N_MEMBERS)]
    group, twins = [], {}
    for i, sc in enumerate(scs):
        kw = dict(iteration_count=iterations, regenerate_noises=int(regen(i)), seed=700 + i)
        if regen(i):
            group.append(_engine(fns, sc, **kw))
            group[-1].generate_noise(5)
            twins[i] = _engine(fns, sc, **kw)
            twins[i].generate_noise(5)
        else:
            group.append(_engine(fns, sc, sc.noise(), **kw))
    hs = _bind(fns, group)
    return scs, group, twins, hs


def _step_and_compare(fns, scs, group, twins, hs, io, iterations, fixed_noise, label):
    ins, outs, _, bufs = io
    assert fns["optimize_batch"](hs, ins, outs, len(group)) == 0
    rtol, atol = (RTOL, ATOL) if iterations == 1 else (RTOL2, ATOL2)
    for i, t in twins.items():
        rt = t.optimize(scs[i].cycle)
        for a, name in zip(bufs[i], ("vx", "vy", "wz")):
            np.testing.assert_allclose(a, getattr(rt, name), rtol=rtol, atol=atol, err_msg=f"{label} robot {i} {name}")
        assert bool(outs[i].fail_flag) == bool(rt.fail_flag), (label, i)
        for p, (a, b) in enumerate(zip(group[i].get_noise(), t.get_noise())):
            assert np.array_equal(a, b), f"{label} robot {i}: noise plane {p} differs in {np.count_nonzero(a != b)} places"
        for e in (group[i], t):
            e.set_control_sequence(rt.vx, rt.vy, rt.wz)
    for i, want in fixed_noise.items():
        for p, (a, b) in enumerate(zip(group[i].get_noise(), want)):
            assert np.array_equal(a, b), f"{label} robot {i}: noise plane {p} of a member without regenerate_noises changed"


@pytest.mark.parametrize("iterations", [1, 2])
def test_regenerating_members_draw_what_unbound_twins_draw(product_fns, iterations):
    """regenerate_noises in a mixed bound group (every other member regenerates), 4 cycles: each regenerating member's
    noise is bit-equal to its unbound twin's after every cycle and its controls match the twin's; the other members'
    noise never changes.  Launches per cycle: 4 per iteration per chunk, one redraw (+ epoch advance) per chunk between
    iterations, and one redraw of all regenerating members behind the last chunk."""
    scs, group, twins, hs = _regen_group(product_fns, iterations, lambda i: i % 2 == 0)
    io = _group_io(scs)
    fixed = {i: group[i].get_noise() for i in range(N_MEMBERS) if i not in twins}
    seen = []
    for cycle in range(4):
        launches0 = _launches(group)
        _step_and_compare(product_fns, scs, group, twins, hs, io, iterations, fixed, f"cycle {cycle}")
        assert _launches(group) - launches0 == 4 * iterations * CHUNKS + 2 * (iterations - 1) * CHUNKS + 2
        seen.append(group[0].get_noise()[0])
    assert not any(np.array_equal(a, b) for a, b in zip(seen, seen[1:]))   # a fresh set every cycle
    for e in group + list(twins.values()):
        e.close()


def test_unbind_continues_the_noise_sequence(product_fns):
    """After mppi_batch_unbind a regenerating member continues on its own exactly where its twin is: the device-side
    stream index and the host's mirror of it stayed in step through the batched cycles."""
    scs, group, twins, hs = _regen_group(product_fns, 2, lambda i: True)
    io = _group_io(scs)
    for cycle in range(2):
        _step_and_compare(product_fns, scs, group, twins, hs, io, 2, {}, f"bound cycle {cycle}")
    assert product_fns["batch_unbind"](group[0].h) == 0
    for i in (0, 37, 65):
        for cycle in range(2):
            rg, rt = group[i].optimize(scs[i].cycle), twins[i].optimize(scs[i].cycle)
            np.testing.assert_allclose(rg.vx, rt.vx, rtol=RTOL2, atol=ATOL2)
            for a, b in zip(group[i].get_noise(), twins[i].get_noise()):
                assert np.array_equal(a, b), f"robot {i} unbound cycle {cycle}"
            for e in (group[i], twins[i]):
                e.set_control_sequence(rt.vx, rt.vy, rt.wz)
        group[i].reset(); twins[i].reset()   # the reset draws the next stream index on both
        assert np.array_equal(group[i].get_noise()[2], twins[i].get_noise()[2])
    for e in group + list(twins.values()):
        e.close()


def test_mixed_iteration_counts_fall_back_one_by_one(product_fns, oracle_fns):
    """Members that differ in iteration_count keep the one-by-one path (mppi_last_error says why) and still give every
    member its oracle's result."""
    scs = [scenarios.config5_robot(r) for r in range(6)]
    for i, sc in enumerate(scs):
        sc.cfg["iteration_count"] = 1 + i % 2
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    orcs = [_engine(oracle_fns, sc, sc.noise()) for sc in scs]
    hs = _bind(product_fns, group)
    ins, outs, keep, bufs = _group_io(scs)
    for cycle in range(2):
        assert product_fns["optimize_batch"](hs, ins, outs, len(scs)) == 0
        assert b"iteration_count" in product_fns["last_error"](group[0].h)
        for i, (sc, o) in enumerate(zip(scs, orcs)):
            ro = o.optimize(sc.cycle)
            _check_against_oracle(f"cycle {cycle} robot {i}", bufs[i], outs[i], group[i], o, ro, sc.cfg["iteration_count"])
            group[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    for e in group + orcs:
        e.close()

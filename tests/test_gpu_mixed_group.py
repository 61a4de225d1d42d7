"""Bound robot groups (mppi_batch_bind) whose members differ in batch_size and time_steps.

Every launch of a chunk spans the chunk's largest member in each grid dimension; each member's job carries its own
extents (rollout blocks, path-cost blocks, weighted-sums chunks, merge blocks, partial-record stride 3T + 2), and the
blocks beyond them return at once.  What goes wrong without that: a small member's surplus blocks write partial records
past its buffer, read another member's stride, or take tickets that fire its last-block election early.

70 members, so that two chunks of 64 run, cycling through five shapes.  1001 x 80 takes the weighted sums' unaligned
branch (B % 4 != 0); 4096 x 24 (most trajectories, shortest horizon) and 600 x 200 (fewest trajectories, longest
horizon) sit next to each other in the first chunk.

- against each member's CPU oracle, with the bars of the existing group tests, and the exact launch count;
- bit for bit against the same scenarios run in homogeneous groups of their own shape (no interference between
  members, no dependence on the grid shape);
- iteration_count = 2 and regenerate_noises (every other member, against unbound twins);
- mppi_optimize_batch_resident against mppi_optimize_batch;
- a member destroyed and re-created with another shape binds back with the others.

Every member runs the same critic list, robot and critic parameters (configs[4] scenarios; every robot stands at the
start of a path of the same length, so the goal gates agree too).  Every chunk therefore needs the same feature set and
runs the same rollout instance in every grouping here, so the bitwise comparisons compare group shapes and not instances.
A chunk whose members need different instances runs the generic one, and nothing promises that it matches an exact
instance bit for bit: only the parity-critical fp32 chains use _rn intrinsics, the rest may be contracted differently.
"""
import numpy as np
import pytest

from mpcholonavigation_b200 import Engine, abi, scenarios

pytestmark = pytest.mark.gpu

RTOL, ATOL, COST_ATOL = 1e-4, 1e-6, 2e-6        # the bars of the iteration_count = 1 group tests
RTOL2, ATOL2 = 1e-3, 1e-5                       # iteration_count = 2 (test_iteration_count_two)
SHAPES = [(2000, 56), (1000, 56), (1001, 80), (4096, 24), (600, 200)]
N_MEMBERS = 70
CHUNKS = 2                                      # of 64 robots


def _scenarios(n=N_MEMBERS, shapes=SHAPES):
    return [scenarios.config5_robot(r, batch=shapes[r % len(shapes)][0], steps=shapes[r % len(shapes)][1]) for r in range(n)]


def _engine(fns, sc, noise=None, **kw):
    e = Engine(fns, **{**sc.cfg, **kw})
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise is not None:
        e.set_noise(*noise)
    return e


def _bind(fns, engines):
    hs = (abi.H * len(engines))(*[e.h for e in engines])
    assert fns["batch_bind"](hs, len(engines)) == 0, fns["last_error"](engines[0].h)
    return hs


def _group_io(scs):
    n = len(scs)
    ins, outs = (abi.CycleIn * n)(), (abi.CycleOut * n)()
    keep, bufs = [], []
    for i, sc in enumerate(scs):
        cin, k = sc.cycle.pack()
        ins[i] = cin
        arrs = [np.empty(sc.cfg["time_steps"], np.float32) for _ in range(3)]
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


def _run_against_oracle(fns, oracle_fns, scs, group, orcs, hs, cycles, iterations, label):
    ins, outs, keep, bufs = _group_io(scs)
    launches0 = _launches(group)
    for cycle in range(cycles):
        assert fns["optimize_batch"](hs, ins, outs, len(scs)) == 0, fns["last_error"](group[0].h)
        for i, (sc, o) in enumerate(zip(scs, orcs)):
            ro = o.optimize(sc.cycle)
            _check_against_oracle(f"{label} cycle {cycle} robot {i} ({sc.name})", bufs[i], outs[i], group[i], o, ro, iterations)
            group[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
    # the batched launches ran: 4 per iteration per chunk (one by one it would be 3 or 1 per robot and iteration)
    assert _launches(group) - launches0 == cycles * CHUNKS * iterations * 4


def test_mixed_shapes_against_the_oracle(product_fns, oracle_fns):
    """Five shapes in one group of 70, 4 cycles: every member's controls, fail flag, furthest point and costs against
    its own oracle, 4 launches per chunk per cycle."""
    scs = _scenarios()
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    orcs = [_engine(oracle_fns, sc, sc.noise()) for sc in scs]
    hs = _bind(product_fns, group)
    _run_against_oracle(product_fns, oracle_fns, scs, group, orcs, hs, 4, 1, "mixed")
    for e in group + orcs:
        e.close()


def test_mixed_group_is_bit_equal_to_homogeneous_groups(product_fns):
    """Each member of the mixed group gives, bit for bit, the controls, fail flag, furthest point, costs and noise of
    the same scenario with the same noise in a homogeneous group of its own shape (14 members each), over 4 cycles in
    which both sides warm-start from their own results."""
    scs = _scenarios()
    mixed = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    hs_mixed = _bind(product_fns, mixed)
    io_mixed = _group_io(scs)
    homog = []
    for s in range(len(SHAPES)):
        idx = list(range(s, N_MEMBERS, len(SHAPES)))
        sub = [scs[i] for i in idx]
        engines = [_engine(product_fns, sc, sc.noise()) for sc in sub]
        homog.append((idx, engines, _bind(product_fns, engines), _group_io(sub)))
    for cycle in range(4):
        ins, outs, _, bufs = io_mixed
        assert product_fns["optimize_batch"](hs_mixed, ins, outs, N_MEMBERS) == 0
        for idx, engines, hs, (hins, houts, _, hbufs) in homog:
            assert product_fns["optimize_batch"](hs, hins, houts, len(idx)) == 0
            for k, i in enumerate(idx):
                label = f"cycle {cycle} robot {i} ({scs[i].name})"
                for a, b, name in zip(bufs[i], hbufs[k], ("vx", "vy", "wz")):
                    assert np.array_equal(a, b), f"{label} {name}: {np.count_nonzero(a != b)} steps differ"
                assert outs[i].fail_flag == houts[k].fail_flag, label
                assert outs[i].furthest_reached_path_point == houts[k].furthest_reached_path_point, label
                cm, ch = mixed[i].get_costs(), engines[k].get_costs()
                assert np.array_equal(cm, ch), f"{label} costs: {np.count_nonzero(cm != ch)} differ"
                for p, (a, b) in enumerate(zip(mixed[i].get_noise(), engines[k].get_noise())):
                    assert np.array_equal(a, b), f"{label} noise plane {p}"
    for _, engines, _, _ in homog:
        for e in engines:
            e.close()
    for e in mixed:
        e.close()


def test_mixed_shapes_iteration_count_two_against_the_oracle(product_fns, oracle_fns):
    """iteration_count = 2 on every member of the mixed group, 3 cycles, against each member's oracle (costs accumulate
    over the iterations, quirk R20); 4 launches per iteration per chunk."""
    scs = _scenarios()
    for sc in scs:
        sc.cfg["iteration_count"] = 2
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    orcs = [_engine(oracle_fns, sc, sc.noise()) for sc in scs]
    hs = _bind(product_fns, group)
    _run_against_oracle(product_fns, oracle_fns, scs, group, orcs, hs, 3, 2, "iteration_count 2")
    for e in group + orcs:
        e.close()


@pytest.mark.parametrize("iterations", [1, 2])
def test_mixed_shapes_regenerating_members_draw_what_unbound_twins_draw(product_fns, iterations):
    """regenerate_noises on every other member of the mixed group (so every shape has members that regenerate and
    members that do not), 3 cycles: after every cycle a regenerating member's noise is bit-equal to its unbound twin's
    and its controls match the twin's; the other members' noise never changes.  The batched redraws are sized for the
    largest regenerating member and cover the smaller ones.  Launches per cycle: 4 per iteration per chunk, a redraw and
    an epoch advance per chunk between iterations, and one redraw + advance of all regenerating members at the end."""
    scs = _scenarios()
    group, twins = [], {}
    for i, sc in enumerate(scs):
        kw = dict(iteration_count=iterations, regenerate_noises=int(i % 2 == 0), seed=900 + i)
        if i % 2 == 0:
            group.append(_engine(product_fns, sc, **kw))
            group[-1].generate_noise(5)
            twins[i] = _engine(product_fns, sc, **kw)
            twins[i].generate_noise(5)
        else:
            group.append(_engine(product_fns, sc, sc.noise(), **kw))
    hs = _bind(product_fns, group)
    ins, outs, _, bufs = _group_io(scs)
    fixed = {i: group[i].get_noise() for i in range(N_MEMBERS) if i not in twins}
    rtol, atol = (RTOL, ATOL) if iterations == 1 else (RTOL2, ATOL2)
    for cycle in range(3):
        launches0 = _launches(group)
        assert product_fns["optimize_batch"](hs, ins, outs, N_MEMBERS) == 0
        assert _launches(group) - launches0 == 4 * iterations * CHUNKS + 2 * (iterations - 1) * CHUNKS + 2
        for i, t in twins.items():
            label = f"cycle {cycle} robot {i} ({scs[i].name})"
            rt = t.optimize(scs[i].cycle)
            for a, name in zip(bufs[i], ("vx", "vy", "wz")):
                np.testing.assert_allclose(a, getattr(rt, name), rtol=rtol, atol=atol, err_msg=f"{label} {name}")
            assert bool(outs[i].fail_flag) == bool(rt.fail_flag), label
            for p, (a, b) in enumerate(zip(group[i].get_noise(), t.get_noise())):
                assert np.array_equal(a, b), f"{label}: noise plane {p} differs in {np.count_nonzero(a != b)} places"
            for e in (group[i], t):
                e.set_control_sequence(rt.vx, rt.vy, rt.wz)
        for i, want in fixed.items():
            for p, (a, b) in enumerate(zip(group[i].get_noise(), want)):
                assert np.array_equal(a, b), f"cycle {cycle} robot {i}: noise plane {p} of a member without regenerate_noises changed"
    for e in group + list(twins.values()):
        e.close()


def test_mixed_shapes_resident_matches_optimize_batch(product_fns):
    """mppi_optimize_batch_resident (the whole group as one chunk) gives bit for bit what mppi_optimize_batch (two
    chunks) gives for the same mixed group, 3 cycles, each side warm-starting from its own results."""
    scs = _scenarios()
    a = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    b = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    hs_a, hs_b = _bind(product_fns, a), _bind(product_fns, b)
    ins, outs_a, _, bufs_a = _group_io(scs)
    _, outs_b, _, bufs_b = _group_io(scs)
    for cycle in range(3):
        assert product_fns["optimize_batch"](hs_a, ins, outs_a, N_MEMBERS) == 0
        for e, sc in zip(b, scs):
            e.upload_cycle(sc.cycle)
        launches0 = _launches(b)
        assert product_fns["optimize_batch_resident"](hs_b, outs_b, N_MEMBERS) == 0
        assert _launches(b) - launches0 == 4
        for i in range(N_MEMBERS):
            label = f"cycle {cycle} robot {i} ({scs[i].name})"
            for x, y, name in zip(bufs_a[i], bufs_b[i], ("vx", "vy", "wz")):
                assert np.array_equal(x, y), f"{label} {name}: {np.count_nonzero(x != y)} steps differ"
            assert outs_a[i].fail_flag == outs_b[i].fail_flag, label
            assert outs_a[i].furthest_reached_path_point == outs_b[i].furthest_reached_path_point, label
            assert np.array_equal(a[i].get_costs(), b[i].get_costs()), f"{label} costs"
    for e in a + b:
        e.close()


def test_rebind_after_a_member_is_recreated_with_another_shape(product_fns, oracle_fns):
    """A dynamic batch_size / time_steps change re-creates a robot's handle; destroying the old one dissolves the group.
    The new handle, of a shape no other member has, binds back with the others, and the group then passes the oracle
    checks of test_mixed_shapes_against_the_oracle."""
    scs = _scenarios()
    group = [_engine(product_fns, sc, sc.noise()) for sc in scs]
    hs = _bind(product_fns, group)
    ins, outs, keep, _ = _group_io(scs)
    assert product_fns["optimize_batch"](hs, ins, outs, N_MEMBERS) == 0
    r = 4                                            # was 600 x 200, next to the 4096 x 24 member
    group[r].close()
    scs[r] = scenarios.config5_robot(r, batch=3000, steps=40)
    group[r] = _engine(product_fns, scs[r], scs[r].noise())
    orcs = [_engine(oracle_fns, sc, sc.noise()) for sc in scs]
    for e, o in zip(group, orcs):                    # the survivors keep their warm start; give the oracles the same
        o.set_control_sequence(*e.get_control_sequence())
    hs = _bind(product_fns, group)
    _run_against_oracle(product_fns, oracle_fns, scs, group, orcs, hs, 2, 1, "rebound")
    for e in group + orcs:
        e.close()

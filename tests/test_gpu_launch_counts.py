"""kernel_launches (mppi_get_profile, bench.py's gpu_launches) for cycles replayed from a captured CUDA graph.

A graph replay counts the launches its capture recorded.  With profiling on and iteration_count = 1 the library skips
the graph and counts every launch as it is issued, so both counts of the same cycle must agree, whichever path the
library picked for it.
"""
import pytest

from mpcholonavigation_b200 import Engine, scenarios

pytestmark = pytest.mark.gpu

STREAM = {"MPPI_STREAM_MIN_BATCH": "64"}

# case: (batch, config overrides, environment, evalControl instead of optimize)
CASES = {
    "fused_1000x56": (1000, {}, {}, False),
    "stream_omni_b_mult4": (2048, {}, STREAM, False),                                  # TMA weighted sums merge
    "stream_ackermann_b_odd": (2050, {"motion_model": "Ackermann"}, STREAM, False),    # separate merge kernel
    "two_kernel": (1000, {}, {"MPPI_FUSED": "0"}, False),
    "regenerate_noises": (1000, {"regenerate_noises": 1, "seed": 11}, {}, False),
    "eval_control_stream": (2048, {}, STREAM, True),
}


def _launches_per_cycle(fns, sc, profiling, eval_control, cycles=3):
    e = Engine(fns, **sc.cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*sc.noise())
    e.set_profiling(profiling)

    def step():
        if eval_control:
            e.eval_control(sc.cycle, True)
        else:
            e.optimize(sc.cycle)

    for _ in range(2):   # the first cycle captures the graph
        step()
    before = e.get_profile()["kernel_launches"]
    for _ in range(cycles):
        step()
    per_cycle = (e.get_profile()["kernel_launches"] - before) / cycles
    e.close()
    return per_cycle


@pytest.mark.parametrize("case", list(CASES))
def test_graph_replay_counts_the_launches_it_runs(product_fns, monkeypatch, case):
    batch, cfg, env, eval_control = CASES[case]
    sc = scenarios.config1(batch=batch)
    sc.cfg.update(cfg, iteration_count=1)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    graph = _launches_per_cycle(product_fns, sc, False, eval_control)
    issued = _launches_per_cycle(product_fns, sc, True, eval_control)
    assert issued > 0
    assert graph == issued, f"{case}: graph replay counts {graph} launches per cycle, issued one by one {issued}"

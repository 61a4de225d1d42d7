"""End-to-end time of a cycle with the costmap in host memory against the same cycle with the map already in device memory
(mppi_set_costmap_residency(MPPI_COSTMAP_DEVICE)), p50 of the host clock around each call (the call returns with the
result in host memory).  The two modes alternate in blocks within one run, so that both see the same machine state.

  1000 x 56, 100 x 100 map (10 KB)        one handle: fused kernel; host mode pulls [record | map] over PCIe itself,
                                          device mode copies the record and runs the path-tables kernel first
  16384 x 56, 2000 x 2000 map (4 MB)      one handle, stream layout: host mode stages and copies 4 MB per cycle
  256 robots x 2000 x 56, one 2000 x 2000 map
                                          a bound group: every member reads the one shared device map, against the same
                                          group with a host copy per member, its slices bound at the 4 MB capacity

usage: python scripts/time_device_costmap.py --out profiles/device_costmap_b200.json [--steps 200]
"""
import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mpcholonavigation_b200 import Engine, abi, load_product, scenarios  # noqa: E402


def _gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in q.split(","))
    return name, power


def _big_map(side=2000):
    """configs[2]'s 400 x 400 inflated-disc map tiled to side x side cells (0.05 m): the robot's surroundings are configs[2]'s"""
    tile = scenarios.config3().cycle.costmap
    reps = -(-side // tile.shape[0])
    return np.ascontiguousarray(np.tile(tile, (reps, reps))[:side, :side])


def _engine(fns, sc, device_map):
    e = Engine(fns, **sc.cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.generate_noise(1)
    e.set_timing(False)
    if device_map:
        e.set_costmap_residency(True)
    return e


def _p50_us(samples):
    return round(float(np.percentile(np.asarray(samples) * 1e6, 50)), 1)


def time_single(fns, sc, steps, warmup, block=20):
    host_cycle = sc.cycle.packed()
    dev_cycle = dataclasses.replace(sc.cycle, costmap=torch.from_numpy(sc.cycle.costmap).cuda()).packed()
    eh, ed = _engine(fns, sc, False), _engine(fns, sc, True)
    for _ in range(warmup):
        eh.optimize(host_cycle)
        ed.optimize(dev_cycle)
    times = {"host": [], "device": []}
    while len(times["device"]) < steps:
        for mode, e, cyc in (("host", eh, host_cycle), ("device", ed, dev_cycle)):
            for _ in range(block):
                t0 = time.perf_counter()
                e.optimize(cyc)
                times[mode].append(time.perf_counter() - t0)
    h2d = {"host": eh.get_profile()["h2d_bytes"], "device": ed.get_profile()["h2d_bytes"]}
    eh.close(); ed.close()
    return {"host_p50_us": _p50_us(times["host"]), "device_p50_us": _p50_us(times["device"]),
            "h2d_bytes_per_cycle": h2d, "cycles_per_mode": len(times["device"])}


def time_group(fns, n, batch, big, steps, warmup):
    T = 56
    scs = [scenarios.config5_robot(r, n_robots=n, batch=batch, steps=T) for r in range(n)]
    big_dev = torch.from_numpy(big).cuda()
    res = {}
    for mode in ("host", "device"):
        es = [_engine(fns, sc, mode == "device") for sc in scs]
        cycles = [dataclasses.replace(sc.cycle, costmap=big if mode == "host" else big_dev) for sc in scs]
        if mode == "host":
            es[0].upload_cycle(cycles[0])   # staging grown to the 4 MB map: the group's slices are bound at that capacity
        hs = (abi.H * n)(*[e.h for e in es])
        assert fns["batch_bind"](hs, n) == 0
        ins, outs, keep = (abi.CycleIn * n)(), (abi.CycleOut * n)(), []
        for i, c in enumerate(cycles):
            cin, k = c.pack()
            ins[i] = cin
            keep.append(k)
        times = []
        for s in range(warmup + steps):
            if mode == "device":
                torch.cuda.current_stream().synchronize()
            t0 = time.perf_counter()
            st = fns["optimize_batch"](hs, ins, outs, n)
            dt = time.perf_counter() - t0
            assert st == 0, fns["last_error"](es[0].h)
            if s >= warmup:
                times.append(dt)
        res[mode + "_p50_us"] = _p50_us(times)
        res[mode + "_h2d_bytes_member0"] = es[0].get_profile()["h2d_bytes"]
        for e in es:
            e.close()
    res["steps_per_mode"] = steps
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--group-steps", type=int, default=30)
    a = ap.parse_args()
    name, power = _gpu_info()
    fns = load_product()
    big = _big_map()
    out = {"gpu": name, "power_limit": power, "timer": "host perf_counter around each call (returns with the result)",
           "cases": {}}
    out["cases"]["omni_1000x56_map100x100"] = time_single(fns, scenarios.config1(), a.steps, a.warmup)
    sc = scenarios.config3()
    sc.cycle = dataclasses.replace(sc.cycle, costmap=big)
    out["cases"]["obstacles_16384x56_map2000x2000"] = time_single(fns, sc, a.steps, a.warmup)
    out["cases"]["robots_256x2000x56_shared_map2000x2000"] = time_group(fns, 256, 2000, big, a.group_steps, 3)
    text = json.dumps(out, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()

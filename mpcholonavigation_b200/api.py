"""numpy-facing wrapper over the C ABI (include/mppi_b200.h).

``Engine`` is written against a table of bound entry points so that the very same driver code can run
the product library (``load_product()``: hand-written sm_100a CUDA kernels, no CPU fallback) and, in
tests only, the CPU oracle.  Method names follow the reference's ``sortham::Optimizer`` members
(nav2_sortham_controller/include/nav2_sortham_controller/optimizer.hpp:72-117).
"""
import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import _abi as abi

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
PRODUCT_LIB = os.path.join(_PKG_DIR, "libmppi_b200.so")


class MppiError(RuntimeError):
    """Raised for any non-OK status from the C ABI (the reference throws std::runtime_error)."""


def load_product(path: Optional[str] = None):
    """dlopen libmppi_b200.so and bind every symbol of the header.  Fails loudly if it is missing:
    there is no Python/CPU fallback for the hot path."""
    path = path or os.environ.get("MPPI_B200_LIB") or PRODUCT_LIB
    if not os.path.exists(path):
        raise MppiError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(path)
    fns = abi.bind(lib, "mppi_", abi.PRODUCT_ONLY)
    fns["_lib"] = lib
    return fns


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(abi.f32p)


def _torch():
    import torch
    return torch


def _is_cuda_tensor(a):
    return getattr(a, "is_cuda", False) and hasattr(a, "data_ptr")


def _sync_device_costmap(cm):
    """The library reads a device costmap without waiting on any stream: the writes torch has queued to it on the
    current stream must be complete before the call."""
    if _is_cuda_tensor(cm):
        _torch().cuda.current_stream(cm.device).synchronize()


@dataclass
class Cycle:
    """Inputs of one Optimizer::evalControl (optimizer.cpp:134-141)."""
    pose: Sequence[float] = (0.0, 0.0, 0.0)          # x, y, yaw
    speed: Sequence[float] = (0.0, 0.0, 0.0)         # vx, vy, wz
    goal: Sequence[float] = (0.0, 0.0)
    goal_checker_xy_tolerance: float = -1.0           # < 0: goal_checker == nullptr
    path_x: np.ndarray = field(default_factory=lambda: np.zeros(1, np.float32))
    path_y: np.ndarray = field(default_factory=lambda: np.zeros(1, np.float32))
    path_yaw: np.ndarray = field(default_factory=lambda: np.zeros(1, np.float32))
    # [size_y, size_x] uint8: a numpy array, or a contiguous CUDA torch tensor for an engine in device-costmap mode
    # (Engine.set_costmap_residency(True))
    costmap: np.ndarray = field(default_factory=lambda: np.zeros((50, 50), np.uint8))
    resolution: float = 0.1
    origin: Sequence[float] = (0.0, 0.0)

    def packed(self):
        """pack() once and keep the result: host buffers that a caller hands over unchanged every cycle (bench e2e leg).
        Call again after modifying the cycle."""
        self._packed = None
        self._packed = self.pack()
        return self

    def pack(self):
        """-> (CycleIn, keepalive list)"""
        cached = getattr(self, "_packed", None)
        if cached is not None:
            _sync_device_costmap(self.costmap)
            return cached
        px, py, pyaw = _f32(self.path_x), _f32(self.path_y), _f32(self.path_yaw)
        assert px.shape == py.shape == pyaw.shape and px.ndim == 1
        if _is_cuda_tensor(self.costmap):
            cm = self.costmap
            if cm.dtype != _torch().uint8 or cm.dim() != 2 or not cm.is_contiguous():
                raise ValueError("a device costmap must be a contiguous 2-D uint8 CUDA tensor")
            cells = C.cast(C.c_void_p(cm.data_ptr()), abi.u8p)
            _sync_device_costmap(cm)
        else:
            cm = np.ascontiguousarray(self.costmap, dtype=np.uint8)
            assert cm.ndim == 2
            cells = cm.ctypes.data_as(abi.u8p)
        cin = abi.CycleIn()
        cin.pose_x, cin.pose_y, cin.pose_yaw = (float(v) for v in self.pose)
        cin.speed_vx, cin.speed_vy, cin.speed_wz = (float(v) for v in self.speed)
        cin.goal_x, cin.goal_y = (float(v) for v in self.goal)
        cin.goal_checker_xy_tolerance = float(self.goal_checker_xy_tolerance)
        cin.path_size = px.shape[0]
        cin.path_x, cin.path_y, cin.path_yaw = _p(px), _p(py), _p(pyaw)
        cin.costmap.cells = cells
        cin.costmap.size_y, cin.costmap.size_x = cm.shape
        cin.costmap.resolution = float(self.resolution)
        cin.costmap.origin_x, cin.costmap.origin_y = (float(v) for v in self.origin)
        return cin, [px, py, pyaw, cm]


@dataclass
class Result:
    vx: np.ndarray
    vy: np.ndarray
    wz: np.ndarray
    fail_flag: bool
    furthest_reached_path_point: Optional[int]
    device_ms: float


def make_config(fns, **kw):
    cfg = abi.Config()
    fns["config_default"](C.byref(cfg))
    for k, v in kw.items():
        if k == "motion_model" and isinstance(v, str):
            v = abi.MOTION_MODELS[v]
        if not hasattr(cfg, k):
            raise KeyError(k)
        setattr(cfg, k, v)
    return cfg


def make_critic(fns, name, **kw):
    d = abi.CriticDesc()
    fns["critic_default"](abi.CRITIC_KINDS[name], C.byref(d))
    for k, v in kw.items():
        if k == "deadband_velocities":
            for i in range(3):
                d.deadband_velocities[i] = float(v[i])
            continue
        if not hasattr(d, k):
            raise KeyError(f"{name}.{k}")
        setattr(d, k, v)
    return d


def make_robot(footprint_xy=(), inscribed_radius=0.0, circumscribed_radius=0.0, inflation_layer_found=False,
               inflation_cost_scaling_factor=10.0, track_unknown=False):
    r = abi.RobotDesc()
    fp = np.asarray(footprint_xy, dtype=np.float64).reshape(-1, 2)
    assert fp.shape[0] <= abi.MAX_FOOTPRINT
    r.footprint_size = fp.shape[0]
    for i in range(fp.shape[0]):
        r.footprint_x[i] = fp[i, 0]
        r.footprint_y[i] = fp[i, 1]
    r.inscribed_radius = inscribed_radius
    r.circumscribed_radius = circumscribed_radius
    r.inflation_layer_found = int(inflation_layer_found)
    r.inflation_cost_scaling_factor = inflation_cost_scaling_factor
    r.track_unknown = int(track_unknown)
    return r


def circle_footprint(radius, n=16):
    """nav2_costmap_2d::makeFootprintFromRadius: 16 points on the circle."""
    a = np.arange(n) * 2.0 * np.pi / n
    return np.stack([radius * np.cos(a), radius * np.sin(a)], axis=1)


class Engine:
    """One ``sortham::Optimizer`` worth of state behind the C ABI."""

    def __init__(self, fns, cfg=None, **cfg_kw):
        self.f = fns
        self.cfg = cfg if cfg is not None else make_config(fns, **cfg_kw)
        self.B, self.T = self.cfg.batch_size, self.cfg.time_steps
        self.h = abi.H()
        self._check(fns["create"](C.byref(self.cfg), C.byref(self.h)), create=True)
        self.n_critics = 0

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, status, create=False):
        if status != abi.MPPI_OK:
            msg = ""
            if "last_error" in self.f and self.h:
                raw = self.f["last_error"](self.h)
                msg = raw.decode() if raw else ""
            raise MppiError(f"mppi status {status}: {msg}")

    def close(self):
        if getattr(self, "h", None):
            self.f["destroy"](self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _planes(self, n=3):
        return [np.empty((self.B, self.T), np.float32) for _ in range(n)]

    # -- configuration ----------------------------------------------------------------------
    def set_critics(self, critics):
        """critics: list of CriticDesc, or of (plugin name, {param: value}) in `critics` list order."""
        descs = []
        for c in critics:
            if isinstance(c, abi.CriticDesc):
                descs.append(c)
            elif isinstance(c, str):
                descs.append(make_critic(self.f, c))
            else:
                descs.append(make_critic(self.f, c[0], **c[1]))
        arr = (abi.CriticDesc * max(1, len(descs)))(*descs)
        self._check(self.f["set_critics"](self.h, arr, len(descs)))
        self.n_critics = len(descs)

    def set_robot(self, robot=None, **kw):
        robot = robot if robot is not None else make_robot(**kw)
        self._check(self.f["set_robot"](self.h, C.byref(robot)))

    def set_speed_limit(self, speed_limit, percentage):
        self._check(self.f["set_speed_limit"](self.h, float(speed_limit), int(bool(percentage))))

    def get_constraints(self):
        out = np.empty(4, np.float32)
        self._check(self.f["get_constraints"](self.h, _p(out)))
        return dict(vx_max=out[0], vx_min=out[1], vy=out[2], wz=out[3])

    def reset(self):
        self._check(self.f["reset"](self.h))

    # -- noise ------------------------------------------------------------------------------
    def set_noise(self, vx, vy, wz):
        vx, wz = _f32(vx), _f32(wz)
        assert vx.shape == (self.B, self.T) and wz.shape == (self.B, self.T)
        vyp = None
        if vy is not None:
            vy = _f32(vy)
            assert vy.shape == (self.B, self.T)
            vyp = _p(vy)
        self._check(self.f["set_noise"](self.h, _p(vx), vyp, _p(wz)))

    def generate_noise(self, stream=0):
        self._check(self.f["generate_noise"](self.h, int(stream)))

    def get_noise(self):
        vx, vy, wz = self._planes()
        self._check(self.f["get_noise"](self.h, _p(vx), _p(vy), _p(wz)))
        return vx, vy, wz

    # -- control sequence -------------------------------------------------------------------
    def set_control_sequence(self, vx, vy, wz):
        vx, vy, wz = _f32(vx), _f32(vy), _f32(wz)
        assert vx.shape == vy.shape == wz.shape == (self.T,)
        self._check(self.f["set_control_sequence"](self.h, _p(vx), _p(vy), _p(wz)))

    def get_control_sequence(self):
        vx, vy, wz = (np.empty(self.T, np.float32) for _ in range(3))
        self._check(self.f["get_control_sequence"](self.h, _p(vx), _p(vy), _p(wz)))
        return vx, vy, wz

    def shift_control_sequence(self):
        self._check(self.f["shift_control_sequence"](self.h))

    # -- hot path ---------------------------------------------------------------------------
    def _out(self):
        vx, vy, wz = (np.empty(self.T, np.float32) for _ in range(3))
        out = abi.CycleOut()
        out.control_vx, out.control_vy, out.control_wz = _p(vx), _p(vy), _p(wz)
        return out, (vx, vy, wz)

    @staticmethod
    def _result(out, arrs):
        f = out.furthest_reached_path_point
        return Result(arrs[0], arrs[1], arrs[2], bool(out.fail_flag), None if f == abi.UINT32_MAX else int(f),
                      float(out.device_ms))

    def optimize(self, cycle: Cycle) -> Result:
        cin, keep = cycle.pack()
        out, arrs = self._out()
        self._check(self.f["optimize"](self.h, C.byref(cin), C.byref(out)))
        del keep
        return self._result(out, arrs)

    def eval_control(self, cycle: Cycle, shift_control_sequence: bool):
        """One attempt of Optimizer::evalControl (optimizer.cpp:134-155): optimize, Savitzky-Golay filter, command
        extraction and control-sequence shift.  Returns ((vx, vy, wz) command, Result)."""
        cin, keep = cycle.pack()
        out, arrs = self._out()
        cmd = np.zeros(3, np.float32)
        self._check(self.f["eval_control"](self.h, C.byref(cin), int(bool(shift_control_sequence)), C.byref(out), _p(cmd)))
        del keep
        return cmd, self._result(out, arrs)

    def set_control_history(self, hist):
        hist = _f32(hist).reshape(12)
        self._check(self.f["set_control_history"](self.h, _p(hist)))

    def get_control_history(self):
        hist = np.zeros(12, np.float32)
        self._check(self.f["get_control_history"](self.h, _p(hist)))
        return hist.reshape(4, 3)

    def upload_cycle(self, cycle: Cycle):
        cin, keep = cycle.pack()
        self._check(self.f["upload_cycle"](self.h, C.byref(cin)))
        del keep

    def optimize_resident(self) -> Result:
        out, arrs = self._out()
        self._check(self.f["optimize_resident"](self.h, C.byref(out)))
        return self._result(out, arrs)

    # -- measurement hooks ------------------------------------------------------------------
    def set_profiling(self, enable=True):
        self._check(self.f["set_profiling"](self.h, int(bool(enable))))

    def register_costmap_memory(self, array):
        """pin the memory of a (C-contiguous uint8) costmap array: cycles whose costmap is this array are uploaded
        straight from it (no staging memcpy).  Keep the array alive until unregister / close."""
        assert array.dtype == np.uint8 and array.flags["C_CONTIGUOUS"]
        self._check(self.f["register_costmap_memory"](self.h, array.ctypes.data, array.nbytes))

    def unregister_costmap_memory(self, array):
        self._check(self.f["unregister_costmap_memory"](self.h, array.ctypes.data))

    def set_costmap_residency(self, device: bool):
        """device=True: the costmap of every cycle is a CUDA tensor on this engine's device, read in place by the kernels
        (no host copy, no upload); False: numpy arrays in host memory (the default)."""
        self._check(self.f["set_costmap_residency"](self.h, abi.COSTMAP_DEVICE if device else abi.COSTMAP_HOST))

    def set_timing(self, enable=True):
        """device_ms of every cycle (two event records + a read-back per call); off: device_ms reads 0"""
        self._check(self.f["set_timing"](self.h, int(bool(enable))))

    def get_profile(self):
        ms = np.zeros(4, np.float32)
        n, h2d, d2h = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self._check(self.f["get_profile"](self.h, _p(ms), C.byref(n), C.byref(h2d), C.byref(d2h)))
        return dict(k2_ms=float(ms[0]), k3_ms=float(ms[1]), exchange_ms=float(ms[2]), span_ms=float(ms[3]),
                    kernel_launches=n.value, h2d_bytes=h2d.value, d2h_bytes=d2h.value)

    # -- sharding ---------------------------------------------------------------------------
    def comm_init(self, unique_id: bytes, rank: int, nranks: int):
        buf = (C.c_uint8 * abi.NCCL_UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self.f["comm_init"](self.h, buf, rank, nranks))

    def comm_mailbox_handle(self) -> bytes:
        """peer-memory exchange, step 1: this rank's 64-byte CUDA IPC handle (all-gather these over any transport)"""
        buf = (C.c_uint8 * abi.IPC_HANDLE_BYTES)()
        self._check(self.f["comm_get_mailbox_handle"](self.h, buf))
        return bytes(buf)

    def comm_connect_peers(self, handles, rank: int, nranks: int):
        """peer-memory exchange, step 2: handles = the nranks handles in rank order"""
        blob = b"".join(handles)
        assert len(blob) == abi.IPC_HANDLE_BYTES * nranks
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._check(self.f["comm_connect_peers"](self.h, buf, rank, nranks))

    # -- introspection ----------------------------------------------------------------------
    def set_outputs(self, trajectories=False, cells=False, critic_costs=False):
        mask = (abi.WANT_TRAJECTORIES if trajectories else 0) | (abi.WANT_CELLS if cells else 0) | \
            (abi.WANT_CRITIC_COSTS if critic_costs else 0)
        if "set_outputs" in self.f:
            self._check(self.f["set_outputs"](self.h, mask))

    def set_visualization(self, trajectory_step, time_step):
        self._check(self.f["set_visualization"](self.h, int(trajectory_step), int(time_step)))
        self._vis = (int(trajectory_step), int(time_step))

    def get_visualization(self):
        ts, s = self._vis
        nb, nt = -(-self.B // ts), -(-self.T // s)
        x, y = np.empty((nb, nt), np.float32), np.empty((nb, nt), np.float32)
        self._check(self.f["get_visualization"](self.h, _p(x), _p(y)))
        return x, y

    def get_trajectories(self):
        x, y, yaw = self._planes()
        self._check(self.f["get_trajectories"](self.h, _p(x), _p(y), _p(yaw)))
        return x, y, yaw

    def get_cells(self):
        cells = np.empty((self.B, self.T), np.int32)
        self._check(self.f["get_cells"](self.h, cells.ctypes.data_as(abi.i32p)))
        return cells

    def get_costs(self):
        c = np.empty(self.B, np.float32)
        self._check(self.f["get_costs"](self.h, _p(c)))
        return c

    def get_critic_costs(self, index):
        c = np.empty(self.B, np.float32)
        self._check(self.f["get_critic_costs"](self.h, int(index), _p(c)))
        return c

    def get_optimized_trajectory(self, pose):
        t = np.empty((self.T, 3), np.float32)
        self._check(self.f["get_optimized_trajectory"](self.h, float(pose[0]), float(pose[1]), float(pose[2]), _p(t)))
        return t

    # -- critic-level / rollout-level entry points --------------------------------------------
    def integrate_state_velocities(self, pose, vx, vy, wz):
        vx, vy, wz = _f32(vx), _f32(vy), _f32(wz)
        assert vx.shape == vy.shape == wz.shape == (self.B, self.T)
        x, y, yaw = self._planes()
        self._check(self.f["integrate_state_velocities"](
            self.h, float(pose[0]), float(pose[1]), float(pose[2]), _p(vx), _p(vy), _p(wz), _p(x), _p(y), _p(yaw)))
        return x, y, yaw

    def score_trajectories(self, cycle: Cycle, vx, vy, wz, x, y, yaw, costs=None, furthest=None):
        """CriticManager::evalTrajectoriesScores on caller-provided State / Trajectories.
        Returns (costs, furthest or None, fail_flag)."""
        arrs = [_f32(a) for a in (vx, vy, wz, x, y, yaw)]
        for a in arrs:
            assert a.shape == (self.B, self.T), a.shape
        costs = np.zeros(self.B, np.float32) if costs is None else _f32(costs).copy()
        fur = C.c_uint32(abi.UINT32_MAX if furthest is None else int(furthest))
        fail = C.c_int32(0)
        cin, keep = cycle.pack()
        self._check(self.f["score_trajectories"](
            self.h, C.byref(cin), *[_p(a) for a in arrs], _p(costs), C.byref(fur), C.byref(fail)))
        del keep
        return costs, (None if fur.value == abi.UINT32_MAX else fur.value), bool(fail.value)


def optimize_sharded(engines, cycle: Cycle) -> Result:
    """mppi_optimize_sharded: the engines are shards of one problem (cfg.shard_offset / shard_total)."""
    e0 = engines[0]
    n = len(engines)
    hs = (abi.H * n)(*[e.h for e in engines])
    cin, keep = cycle.pack()
    out, arrs = e0._out()
    status = e0.f["optimize_sharded"](hs, n, C.byref(cin), C.byref(out))
    del keep
    if status != abi.MPPI_OK:
        msgs = [e.f["last_error"](e.h).decode() for e in engines]
        raise MppiError(f"mppi status {status}: {msgs}")
    return Engine._result(out, arrs)


def optimize_group_device(engines, state, tolerance, path_size, path, maps):
    """mppi_optimize_group_device: one cycle of a bound group (``engines`` in bind order, every one in device-costmap
    mode) whose inputs are CUDA tensors on the group's device, one row per member:
    state float64 [n, 8] (pose x, y, yaw, speed vx, vy, wz, goal x, y), tolerance float64 [n] (< 0: no goal checker),
    path_size int32 [n], path float32 [n, 3, stride] (x, y, yaw).  maps: per member (uint8 CUDA tensor [size_y, size_x],
    resolution, (origin_x, origin_y)).  The records are built on the device; returns a list of Result."""
    torch = _torch()
    n = len(engines)
    e0 = engines[0]
    tensors = {"state": (state, torch.float64, (n, 8)), "tolerance": (tolerance, torch.float64, (n,)),
               "path_size": (path_size, torch.int32, (n,)), "path": (path, torch.float32, None)}
    for name, (t, dtype, shape) in tensors.items():
        if not _is_cuda_tensor(t) or t.dtype != dtype or not t.is_contiguous() or (shape and tuple(t.shape) != shape):
            raise ValueError(f"{name}: a contiguous {dtype} CUDA tensor{' of shape ' + str(shape) if shape else ''} is expected")
    if path.dim() != 3 or path.shape[0] != n or path.shape[1] != 3:
        raise ValueError("path: [n, 3, stride] expected")
    gi = abi.GroupInputs()
    gi.state, gi.goal_checker_xy_tolerance = state.data_ptr(), tolerance.data_ptr()
    gi.path_size, gi.path, gi.path_stride = path_size.data_ptr(), path.data_ptr(), path.shape[2]
    cms = (abi.Costmap * n)()
    for i, (cells, resolution, origin) in enumerate(maps):
        if not _is_cuda_tensor(cells) or cells.dtype != torch.uint8 or cells.dim() != 2 or not cells.is_contiguous():
            raise ValueError("maps: contiguous 2-D uint8 CUDA tensors expected")
        cms[i].cells = C.cast(C.c_void_p(cells.data_ptr()), abi.u8p)
        cms[i].size_y, cms[i].size_x = cells.shape
        cms[i].resolution = float(resolution)
        cms[i].origin_x, cms[i].origin_y = (float(v) for v in origin)
    # the library reads the inputs without waiting on any stream: torch's queued writes must be complete
    for device in {t.device for t in [state, tolerance, path_size, path] + [m[0] for m in maps]}:
        torch.cuda.current_stream(device).synchronize()
    outs = (abi.CycleOut * n)()
    arrs = []
    for i, e in enumerate(engines):
        o, a = e._out()
        outs[i] = o
        arrs.append(a)
    hs = (abi.H * n)(*[e.h for e in engines])
    e0._check(e0.f["optimize_group_device"](hs, n, C.byref(gi), cms, outs))
    return [Engine._result(outs[i], arrs[i]) for i in range(n)]
